// cg_cloud.cu -- point-cloud front end of the per-object grasp stage (float64 throughout).
//
// Replaces the open3d / scipy.spatial.cKDTree work of run_grasp_simulation.py:113-139,171-175,198-211,245-251:
//   * cg_cloud: an occupied-cell grid over a resident (N,3) cloud.  Points are sorted by a hierarchical cell key
//     (coarse cell = 8x8x8 fine cells in the high bits, the fine cell inside it in the low 9 bits), so the points of one
//     fine cell and of one coarse cell are both contiguous ranges.  Two open-addressing hash tables map an occupied
//     fine / coarse cell to its [start, end) range.  Memory is O(N) whatever the bounding-box volume.
//   * nearest neighbour (cKDTree.query, k=1): exact ring search over coarse cells around the (clamped) query cell, every
//     cell pruned by its box distance, the search stopped by the box distance of the unvisited part of the grid.  Queries
//     outside the cloud's box start at the nearest boundary cell, so far queries cost the lateral rings only.
//   * any-within-radius: same pruning with a fixed bound r and an early exit on the first hit (fine cells when the
//     ball spans at most 64 of them, coarse cells otherwise).
//   * normals of the indexed points: open3d EstimateNormals(KDTreeSearchParamHybrid(radius, max_nn)) restated -- the
//     max_nn nearest with d^2 < r^2 (scipy's distance_upper_bound rule, the point itself included, ties to the lower
//     index), the cumulant covariance, the eigenvector of the smallest eigenvalue (cyclic Jacobi), (0,0,1) with fewer
//     than 3 neighbours -- fused with Utils.py:205-213 correct_pcd_normal_direction.  One warp per 32 consecutive
//     (cell-ordered) points: the warp finds the neighbours of each of the 32 in turn, keeping the sorted top-k list one
//     slot per lane; lane j keeps point j's covariance, then all 32 lanes run their Jacobi at once.
//   * voxel down-sampling: open3d VoxelDownSample restated -- voxel_min_bound = min - 0.5*voxel, index =
//     floor((p - voxel_min_bound) / voxel), per-voxel sums in INPUT order divided by the count (normals not
//     re-normalised).  Output in ascending voxel index order (x, then y, then z); open3d emits its hash-map order.
// Distances are ((dx*dx + dy*dy) + dz*dz) without contraction, the order scipy's kd-tree accumulates them in.
#include <cub/cub.cuh>
#include <algorithm>
#include <climits>
#include <cmath>

#include "cg_common.cuh"

namespace {

constexpr unsigned long long EMPTY_KEY = ~0ull;
constexpr int CBITS = 3;                 // coarse cell = 2^3 fine cells per axis
constexpr int MAX_AXIS_CELLS = 1 << 21;  // fine cells per axis (key = 3 x 18 coarse bits + 9 local bits)

struct HashE {
  unsigned long long key;
  int start, end;
};

}  // namespace

struct cg_cloud {
  cg_ctx *ctx = nullptr;
  int N = 0;
  double cell = 0.0;
  double org[3] = {0, 0, 0};    // bounding-box min = fine cell (0,0,0) corner
  double bmax[3] = {0, 0, 0};
  int dims[3] = {0, 0, 0};      // fine cells per axis
  int cdims[3] = {0, 0, 0};     // coarse cells per axis
  double *spts = nullptr;       // (N,3) points in cell-key order
  int32_t *sidx = nullptr;      // original index of spts[s]
  HashE *fine = nullptr, *coarse = nullptr;
  uint32_t fmask = 0, cmask = 0;
};

namespace {

struct Grid {
  const double *pts;
  const int32_t *idx;
  const HashE *fine, *coarse;
  uint32_t fmask, cmask;
  int N;
  double cell, ccell;
  double org[3], bmax[3];
  int dims[3], cdims[3];
};

Grid view(const cg_cloud *c) {
  Grid g;
  g.pts = c->spts; g.idx = c->sidx; g.fine = c->fine; g.coarse = c->coarse;
  g.fmask = c->fmask; g.cmask = c->cmask; g.N = c->N;
  g.cell = c->cell; g.ccell = c->cell * (1 << CBITS);
  for (int a = 0; a < 3; a++) {
    g.org[a] = c->org[a]; g.bmax[a] = c->bmax[a]; g.dims[a] = c->dims[a]; g.cdims[a] = c->cdims[a];
  }
  return g;
}

__host__ __device__ __forceinline__ unsigned long long coarse_lin(const int *cd, int cx, int cy, int cz) {
  return ((unsigned long long)cx * cd[1] + cy) * cd[2] + cz;
}
__host__ __device__ __forceinline__ unsigned long long fine_key(const int *cd, int ix, int iy, int iz) {
  return (coarse_lin(cd, ix >> CBITS, iy >> CBITS, iz >> CBITS) << (3 * CBITS)) |
         (unsigned long long)(((ix & 7) << 6) | ((iy & 7) << 3) | (iz & 7));
}

__device__ __forceinline__ uint32_t hash64(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull;
  k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull;
  k ^= k >> 33;
  return (uint32_t)k;
}

__device__ __forceinline__ bool lookup(const HashE *t, uint32_t mask, unsigned long long key, int &s, int &e) {
  uint32_t h = hash64(key) & mask;
  while (true) {
    const unsigned long long k = t[h].key;
    if (k == key) { s = t[h].start; e = t[h].end; return true; }
    if (k == EMPTY_KEY) return false;
    h = (h + 1) & mask;
  }
}

__device__ __forceinline__ double sqdist(double qx, double qy, double qz, const double *p) {
  const double dx = __dsub_rn(qx, p[0]), dy = __dsub_rn(qy, p[1]), dz = __dsub_rn(qz, p[2]);
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// lower bound of |q - x| over x in [lo, hi] along one axis; the slack absorbs the rounding of cell boundaries so the
// bound never exceeds the distance a point of the cell is computed at
__device__ __forceinline__ double gap(double q, double lo, double hi, double slack) {
  const double d = q < lo ? lo - q : (q > hi ? q - hi : 0.0);
  return fmax(d - slack, 0.0);
}
__device__ __forceinline__ double box_d2(const double *q, const double *lo, const double *hi, double slack) {
  const double gx = gap(q[0], lo[0], hi[0], slack), gy = gap(q[1], lo[1], hi[1], slack), gz = gap(q[2], lo[2], hi[2], slack);
  return gx * gx + gy * gy + gz * gz;
}

// cell of coordinate v on a grid of n cells (clamped: queries outside the box map to the nearest boundary cell)
__device__ __forceinline__ int cell_of(double v, double org, double size, int n) {
  double f = floor((v - org) / size);
  f = fmin(fmax(f, 0.0), (double)(n - 1));
  return (int)f;
}

__device__ __forceinline__ bool better(double d, int i, double bd, int bi) { return d < bd || (d == bd && i < bi); }

// ---- index construction ------------------------------------------------------------------------------------------

__device__ __forceinline__ unsigned long long dkey(double v) {   // order-preserving double -> uint64
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__host__ double key2d(unsigned long long k) {
  const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  double v;
  memcpy(&v, &b, 8);
  return v;
}

// bb[0..2] = min keys (init ~0), bb[3..5] = max keys (init 0), bb[6] = non-finite flag
__global__ void bbox_kernel(const double *__restrict__ pts, int N, unsigned long long *bb) {
  unsigned long long mn[3] = {EMPTY_KEY, EMPTY_KEY, EMPTY_KEY}, mx[3] = {0, 0, 0};
  unsigned long long bad = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x)
    for (int a = 0; a < 3; a++) {
      const double v = pts[3 * i + a];
      if (!isfinite(v)) { bad = 1; continue; }
      const unsigned long long k = dkey(v);
      mn[a] = k < mn[a] ? k : mn[a];
      mx[a] = k > mx[a] ? k : mx[a];
    }
  for (int a = 0; a < 3; a++)
    for (int o = 16; o; o >>= 1) {
      const unsigned long long m = __shfl_xor_sync(0xffffffffu, mn[a], o), M = __shfl_xor_sync(0xffffffffu, mx[a], o);
      mn[a] = m < mn[a] ? m : mn[a];
      mx[a] = M > mx[a] ? M : mx[a];
    }
  bad = __any_sync(0xffffffffu, bad != 0);
  if ((threadIdx.x & 31) == 0) {
    for (int a = 0; a < 3; a++) { atomicMin(&bb[a], mn[a]); atomicMax(&bb[3 + a], mx[a]); }
    if (bad) atomicOr(&bb[6], 1ull);
  }
}

__global__ void cell_key_kernel(const double *__restrict__ pts, int N, Grid g, unsigned long long *__restrict__ keys,
                                int32_t *__restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int c[3];
  for (int a = 0; a < 3; a++) c[a] = cell_of(pts[3 * i + a], g.org[a], g.cell, g.dims[a]);
  keys[i] = fine_key(g.cdims, c[0], c[1], c[2]);
  vals[i] = i;
}

__global__ void gather_kernel(const double *__restrict__ pts, const int32_t *__restrict__ order, int N,
                              double *__restrict__ spts, int32_t *__restrict__ sidx, const unsigned long long *__restrict__ keys,
                              unsigned long long *__restrict__ ckeys) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= N) return;
  const int i = order[s];
  spts[3 * s] = pts[3 * i];
  spts[3 * s + 1] = pts[3 * i + 1];
  spts[3 * s + 2] = pts[3 * i + 2];
  sidx[s] = i;
  ckeys[s] = keys[s] >> (3 * CBITS);
}

__global__ void hash_insert_kernel(const unsigned long long *__restrict__ uniq, const int *__restrict__ counts,
                                   const int *__restrict__ starts, const int *__restrict__ nruns, HashE *table, uint32_t mask) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= *nruns) return;
  const unsigned long long key = uniq[r];
  uint32_t h = hash64(key) & mask;
  while (atomicCAS(&table[h].key, EMPTY_KEY, key) != EMPTY_KEY) h = (h + 1) & mask;
  table[h].start = starts[r];
  table[h].end = starts[r] + counts[r];
}

// ---- nearest neighbour ---------------------------------------------------------------------------------------------

__device__ void scan_range(const Grid &g, const double *q, int s, int e, double &best, int &bi) {
  for (int j = s; j < e; j++) {
    const double d = sqdist(q[0], q[1], q[2], g.pts + 3 * j);
    const int id = g.idx[j];
    if (better(d, id, best, bi)) { best = d; bi = id; }
  }
}

__device__ void visit_coarse(const Grid &g, const double *q, int x, int y, int z, double slack, double &best, int &bi) {
  const double lo[3] = {g.org[0] + x * g.ccell, g.org[1] + y * g.ccell, g.org[2] + z * g.ccell};
  const double hi[3] = {lo[0] + g.ccell, lo[1] + g.ccell, lo[2] + g.ccell};
  if (box_d2(q, lo, hi, slack) > best) return;
  int s, e;
  if (!lookup(g.coarse, g.cmask, coarse_lin(g.cdims, x, y, z), s, e)) return;
  scan_range(g, q, s, e, best, bi);
}

__global__ void nearest_kernel(Grid g, const double *__restrict__ qs, int Q, double *__restrict__ out_d,
                               int32_t *__restrict__ out_i) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= Q) return;
  const double q[3] = {qs[3 * t], qs[3 * t + 1], qs[3 * t + 2]};
  double best = INFINITY;
  int bi = INT_MAX;
  if (g.N > 0 && isfinite(q[0]) && isfinite(q[1]) && isfinite(q[2])) {
    const double slack = 1e-9 * g.ccell;
    int c[3];
    for (int a = 0; a < 3; a++) c[a] = cell_of(q[a], g.org[a], g.ccell, g.cdims[a]);
    for (int R = 0;; R++) {
      if (R > 0) {   // stop once every unvisited coarse cell (the slabs outside the visited cube) is farther than best
        double lb = INFINITY;
        bool open = false;
        for (int a = 0; a < 3; a++) {
          double lo[3] = {g.org[0], g.org[1], g.org[2]}, hi[3] = {g.bmax[0], g.bmax[1], g.bmax[2]};
          if (c[a] - (R - 1) > 0) {
            hi[a] = g.org[a] + (c[a] - R + 1) * g.ccell;
            lb = fmin(lb, box_d2(q, lo, hi, slack));
            open = true;
            hi[a] = g.bmax[a];
          }
          if (c[a] + (R - 1) < g.cdims[a] - 1) {
            lo[a] = g.org[a] + (c[a] + R) * g.ccell;
            lb = fmin(lb, box_d2(q, lo, hi, slack));
            open = true;
          }
        }
        if (!open || lb > best) break;
      }
      const int x0 = max(c[0] - R, 0), x1 = min(c[0] + R, g.cdims[0] - 1);
      const int y0 = max(c[1] - R, 0), y1 = min(c[1] + R, g.cdims[1] - 1);
      for (int x = x0; x <= x1; x++)
        for (int y = y0; y <= y1; y++) {
          if (R == 0 || x == c[0] - R || x == c[0] + R || y == c[1] - R || y == c[1] + R) {
            for (int z = max(c[2] - R, 0); z <= min(c[2] + R, g.cdims[2] - 1); z++) visit_coarse(g, q, x, y, z, slack, best, bi);
          } else {
            if (c[2] - R >= 0) visit_coarse(g, q, x, y, c[2] - R, slack, best, bi);
            if (c[2] + R < g.cdims[2]) visit_coarse(g, q, x, y, c[2] + R, slack, best, bi);
          }
        }
    }
  }
  out_d[t] = sqrt(best);
  out_i[t] = bi == INT_MAX ? g.N : bi;   // no point: cKDTree's "missing neighbour" index n
}

// ---- any point within r ----------------------------------------------------------------------------------------------

__device__ bool hit_range(const Grid &g, const double *q, int s, int e, double r) {
  for (int j = s; j < e; j++)
    if (sqrt(sqdist(q[0], q[1], q[2], g.pts + 3 * j)) <= r) return true;
  return false;
}

__global__ void any_within_kernel(Grid g, const double *__restrict__ qs, int Q, double r, uint8_t *__restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= Q) return;
  const double q[3] = {qs[3 * t], qs[3 * t + 1], qs[3 * t + 2]};
  uint8_t hit = 0;
  const double r2 = r * r * (1.0 + 1e-12);
  const double slack = 1e-9 * g.ccell;
  if (g.N > 0 && isfinite(q[0]) && isfinite(q[1]) && isfinite(q[2]) && box_d2(q, g.org, g.bmax, slack) <= r2) {
    int lo[3], hi[3];
    long n = 1;
    for (int a = 0; a < 3; a++) {
      lo[a] = cell_of(q[a] - r, g.org[a], g.cell, g.dims[a]);
      hi[a] = cell_of(q[a] + r, g.org[a], g.cell, g.dims[a]);
      n *= hi[a] - lo[a] + 1;
    }
    const bool fine = n <= 64;
    const double size = fine ? g.cell : g.ccell;
    if (!fine)
      for (int a = 0; a < 3; a++) { lo[a] >>= CBITS; hi[a] >>= CBITS; }
    for (int x = lo[0]; x <= hi[0] && !hit; x++)
      for (int y = lo[1]; y <= hi[1] && !hit; y++)
        for (int z = lo[2]; z <= hi[2] && !hit; z++) {
          const double blo[3] = {g.org[0] + x * size, g.org[1] + y * size, g.org[2] + z * size};
          const double bhi[3] = {blo[0] + size, blo[1] + size, blo[2] + size};
          if (box_d2(q, blo, bhi, slack) > r2) continue;
          int s, e;
          const bool occ = fine ? lookup(g.fine, g.fmask, fine_key(g.cdims, x, y, z), s, e)
                                : lookup(g.coarse, g.cmask, coarse_lin(g.cdims, x, y, z), s, e);
          if (occ && hit_range(g, q, s, e, r)) hit = 1;
        }
  }
  out[t] = hit;
}

// ---- normals -------------------------------------------------------------------------------------------------------

constexpr int NW = 8;   // warps per block in normals_kernel

// one cyclic-Jacobi rotation in the (p, q) plane of the symmetric 3x3 A (row-major), accumulated into V's columns
template <int p, int q, int r>
__device__ __forceinline__ void jrot(double *A, double *V) {
  const double apq = A[p * 3 + q];
  if (apq == 0.0) return;
  const double theta = (A[q * 3 + q] - A[p * 3 + p]) / (2.0 * apq);
  double t = fabs(theta) > 1e150 ? 0.5 / theta : 1.0 / (fabs(theta) + sqrt(theta * theta + 1.0));
  if (theta < 0.0 && fabs(theta) <= 1e150) t = -t;
  const double c = 1.0 / sqrt(t * t + 1.0), s = t * c, tau = s / (1.0 + c);
  A[p * 3 + p] -= t * apq;
  A[q * 3 + q] += t * apq;
  A[p * 3 + q] = A[q * 3 + p] = 0.0;
  const double g = A[r * 3 + p], h = A[r * 3 + q];
  A[r * 3 + p] = A[p * 3 + r] = g - s * (h + g * tau);
  A[r * 3 + q] = A[q * 3 + r] = h + s * (g - h * tau);
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const double vg = V[k * 3 + p], vh = V[k * 3 + q];
    V[k * 3 + p] = vg - s * (vh + vg * tau);
    V[k * 3 + q] = vh + s * (vg - vh * tau);
  }
}

// eigenvector of the smallest eigenvalue of the symmetric covariance (c = xx, xy, xz, yy, yz, zz)
__device__ void smallest_eigvec(const double *c, double *n) {
  double A[9] = {c[0], c[1], c[2], c[1], c[3], c[4], c[2], c[4], c[5]};
  double V[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  for (int sweep = 0; sweep < 50; sweep++) {
    const double off = A[1] * A[1] + A[2] * A[2] + A[5] * A[5];
    const double diag = A[0] * A[0] + A[4] * A[4] + A[8] * A[8];
    if (off == 0.0 || off <= 1e-36 * diag) break;
    jrot<0, 1, 2>(A, V);
    jrot<0, 2, 1>(A, V);
    jrot<1, 2, 0>(A, V);
  }
  int k = 0;
  if (A[4] < A[k * 4]) k = 1;
  if (A[8] < A[k * 4]) k = 2;
  n[0] = V[k]; n[1] = V[3 + k]; n[2] = V[6 + k];
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(NW * 32) normals_kernel(Grid g, double r, double r2, int K, double vpx, double vpy,
                                                          double vpz, double *__restrict__ out, int32_t *__restrict__ nbr) {
  __shared__ int s_pref[NW][32], s_start[NW][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int base = (blockIdx.x * NW + w) * 32;
  if (base >= g.N) return;
  double mc[6] = {0, 0, 0, 0, 0, 0};
  int mn = 0;
  const int nj = min(32, g.N - base);
  for (int j = 0; j < nj; j++) {
    const double *p = g.pts + 3 * (base + j);
    const double px = p[0], py = p[1], pz = p[2];
    const double q[3] = {px, py, pz};
    int lo[3], ext[3];
    for (int a = 0; a < 3; a++) {
      lo[a] = cell_of(q[a] - r, g.org[a], g.cell, g.dims[a]);
      ext[a] = cell_of(q[a] + r, g.org[a], g.cell, g.dims[a]) - lo[a] + 1;
    }
    const int ncell = ext[0] * ext[1] * ext[2];
    // sorted top-K list, slot = lane: (distance^2, original index, coordinates)
    double ld = INFINITY, lx = 0, ly = 0, lz = 0;
    int li = INT_MAX;
    double kd = INFINITY;
    int ki = INT_MAX;
    for (int cb = 0; cb < ncell; cb += 32) {
      const int t = cb + lane;
      int cs = 0, ce = 0;
      if (t < ncell) {
        const int x = lo[0] + t / (ext[1] * ext[2]), y = lo[1] + (t / ext[2]) % ext[1], z = lo[2] + t % ext[2];
        const double blo[3] = {g.org[0] + x * g.cell, g.org[1] + y * g.cell, g.org[2] + z * g.cell};
        const double bhi[3] = {blo[0] + g.cell, blo[1] + g.cell, blo[2] + g.cell};
        if (box_d2(q, blo, bhi, 1e-9 * g.cell) < r2 * (1.0 + 1e-12)) lookup(g.fine, g.fmask, fine_key(g.cdims, x, y, z), cs, ce);
      }
      int pref = ce - cs;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, pref, o);
        if (lane >= o) pref += v;
      }
      s_pref[w][lane] = pref;
      s_start[w][lane] = cs;
      __syncwarp();
      const int total = __shfl_sync(0xffffffffu, pref, 31);
      for (int b2 = 0; b2 < total; b2 += 32) {
        const int tt = b2 + lane;
        double d = INFINITY, cx = 0, cy = 0, cz = 0;
        int id = INT_MAX;
        if (tt < total) {
          int o = 0;   // first cell whose inclusive prefix exceeds tt
#pragma unroll
          for (int step = 16; step; step >>= 1)
            if (s_pref[w][o + step - 1] <= tt) o += step;
          const int pos = s_start[w][o] + tt - (o ? s_pref[w][o - 1] : 0);
          cx = g.pts[3 * pos]; cy = g.pts[3 * pos + 1]; cz = g.pts[3 * pos + 2];
          const double dx = __dsub_rn(px, cx), dy = __dsub_rn(py, cy), dz = __dsub_rn(pz, cz);
          d = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
          id = g.idx[pos];
        }
        unsigned mask = __ballot_sync(0xffffffffu, d < r2 && better(d, id, kd, ki));
        while (mask) {
          const int src = __ffs(mask) - 1;
          const double nd = __shfl_sync(0xffffffffu, d, src);
          const int ni = __shfl_sync(0xffffffffu, id, src);
          const double nx = __shfl_sync(0xffffffffu, cx, src), ny = __shfl_sync(0xffffffffu, cy, src),
                       nz = __shfl_sync(0xffffffffu, cz, src);
          const int at = __popc(__ballot_sync(0xffffffffu, better(ld, li, nd, ni)));
          const double ud = __shfl_up_sync(0xffffffffu, ld, 1), ux = __shfl_up_sync(0xffffffffu, lx, 1),
                       uy = __shfl_up_sync(0xffffffffu, ly, 1), uz = __shfl_up_sync(0xffffffffu, lz, 1);
          const int ui = __shfl_up_sync(0xffffffffu, li, 1);
          if (lane == at) { ld = nd; li = ni; lx = nx; ly = ny; lz = nz; }
          else if (lane > at) { ld = ud; li = ui; lx = ux; ly = uy; lz = uz; }
          kd = __shfl_sync(0xffffffffu, ld, K - 1);
          ki = __shfl_sync(0xffffffffu, li, K - 1);
          mask &= ~(1u << src);
          mask &= __ballot_sync(0xffffffffu, better(d, id, kd, ki));
        }
      }
      __syncwarp();
    }
    const bool mine = lane < K && ld < r2;
    const int n = __popc(__ballot_sync(0xffffffffu, mine));
    if (nbr && lane < K) nbr[(size_t)g.idx[base + j] * K + lane] = mine ? li : g.N;
    if (n >= 3) {   // open3d's cumulant form of the covariance
      const double x = mine ? lx : 0.0, y = mine ? ly : 0.0, z = mine ? lz : 0.0;
      const double inv = (double)n;
      const double c0 = warp_sum(x) / inv, c1 = warp_sum(y) / inv, c2 = warp_sum(z) / inv;
      const double c3 = warp_sum(x * x) / inv, c4 = warp_sum(x * y) / inv, c5 = warp_sum(x * z) / inv;
      const double c6 = warp_sum(y * y) / inv, c7 = warp_sum(y * z) / inv, c8 = warp_sum(z * z) / inv;
      if (lane == j) {
        mc[0] = c3 - c0 * c0; mc[1] = c4 - c0 * c1; mc[2] = c5 - c0 * c2;
        mc[3] = c6 - c1 * c1; mc[4] = c7 - c1 * c2; mc[5] = c8 - c2 * c2;
      }
    }
    if (lane == j) mn = n;
  }
  if (lane >= nj) return;
  const int s = base + lane;
  double nv[3] = {0.0, 0.0, 1.0};
  if (mn >= 3) {
    smallest_eigvec(mc, nv);
    if (nv[0] == 0.0 && nv[1] == 0.0 && nv[2] == 0.0) { nv[2] = 1.0; }
  }
  // Utils.py:205-213, numpy's operation order
  const double *p = g.pts + 3 * s;
  double vx = __dsub_rn(vpx, p[0]), vy = __dsub_rn(vpy, p[1]), vz = __dsub_rn(vpz, p[2]);
  const double vn = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy)), __dmul_rn(vz, vz)));
  vx = vx / vn; vy = vy / vn; vz = vz / vn;
  const double nn = __dadd_rn(sqrt(__dadd_rn(__dadd_rn(__dmul_rn(nv[0], nv[0]), __dmul_rn(nv[1], nv[1])), __dmul_rn(nv[2], nv[2]))), 1e-10);
  double ox = nv[0] / nn, oy = nv[1] / nn, oz = nv[2] / nn;
  const double dot = __dadd_rn(__dadd_rn(__dmul_rn(vx, ox), __dmul_rn(vy, oy)), __dmul_rn(vz, oz));
  if (dot < 0.0) { ox = -ox; oy = -oy; oz = -oz; }
  const int i = g.idx[s];
  out[3 * i] = ox;
  out[3 * i + 1] = oy;
  out[3 * i + 2] = oz;
}

// ---- voxel down-sampling -------------------------------------------------------------------------------------------

__global__ void voxel_index_kernel(const double *__restrict__ pts, int N, double mx, double my, double mz, double voxel,
                                   int32_t *__restrict__ vi, int32_t *__restrict__ order) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  vi[3 * i] = (int)floor(__ddiv_rn(__dsub_rn(pts[3 * i], mx), voxel));
  vi[3 * i + 1] = (int)floor(__ddiv_rn(__dsub_rn(pts[3 * i + 1], my), voxel));
  vi[3 * i + 2] = (int)floor(__ddiv_rn(__dsub_rn(pts[3 * i + 2], mz), voxel));
  order[i] = i;
}

// sort key of one LSD pass: the axes [a0, 3) packed with `bits[a]` bits each, x most significant
__global__ void voxel_key_kernel(const int32_t *__restrict__ vi, const int32_t *__restrict__ order, int N, int a0, int a1,
                                 int b1, int b2, unsigned long long *__restrict__ keys) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= N) return;
  const int32_t *v = vi + 3 * order[s];
  unsigned long long k = 0;
  for (int a = a0; a < a1; a++) k = (k << (a == 1 ? b1 : a == 2 ? b2 : 0)) | (unsigned long long)v[a];
  keys[s] = k;
}

__global__ void voxel_head_kernel(const int32_t *__restrict__ vi, const int32_t *__restrict__ order, int N,
                                  int32_t *__restrict__ head) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= N) return;
  int h = 1;
  if (s > 0) {
    const int32_t *a = vi + 3 * order[s], *b = vi + 3 * order[s - 1];
    h = (a[0] != b[0]) || (a[1] != b[1]) || (a[2] != b[2]);
  }
  head[s] = h;
}

__global__ void voxel_seg_kernel(const int32_t *__restrict__ head, const int32_t *__restrict__ slot, int N,
                                 int32_t *__restrict__ seg_start, int32_t *__restrict__ count) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= N) return;
  if (head[s]) seg_start[slot[s]] = s;
  if (s == N - 1) *count = slot[s] + head[s];
}

__global__ void voxel_mean_kernel(const double *__restrict__ pts, const double *__restrict__ nrm,
                                  const int32_t *__restrict__ order, const int32_t *__restrict__ seg_start,
                                  const int32_t *__restrict__ count, int N, double *__restrict__ out_p,
                                  double *__restrict__ out_n) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  const int nv = *count;
  if (v >= nv) return;
  const int a = seg_start[v], b = v + 1 < nv ? seg_start[v + 1] : N;
  double sp[3] = {0.0, 0.0, 0.0}, sn[3] = {0.0, 0.0, 0.0};
  for (int s = a; s < b; s++) {   // input order: the sorts are stable over an identity permutation
    const int i = order[s];
    for (int k = 0; k < 3; k++) sp[k] = __dadd_rn(sp[k], pts[3 * i + k]);
    if (nrm)
      for (int k = 0; k < 3; k++) sn[k] = __dadd_rn(sn[k], nrm[3 * i + k]);
  }
  const double c = (double)(b - a);
  for (int k = 0; k < 3; k++) out_p[3 * v + k] = __ddiv_rn(sp[k], c);
  if (nrm)
    for (int k = 0; k < 3; k++) out_n[3 * v + k] = __ddiv_rn(sn[k], c);
}

inline unsigned blocks(long n, int t) { return (unsigned)((n + t - 1) / t); }

int bits_for(long v) {   // bits needed to hold 0..v
  int b = 0;
  while (b < 63 && (1L << b) <= v) b++;
  return b;
}

// bounding box of (N,3) points into host doubles; CG_EINVAL on non-finite input.  Synchronises the context stream.
int device_bbox(cg_ctx *ctx, const double *pts, int N, unsigned long long *bb_dev, double *mn, double *mx) {
  CG_CUDA(ctx, cudaMemsetAsync(bb_dev, 0xff, 3 * sizeof(unsigned long long), ctx->stream));
  CG_CUDA(ctx, cudaMemsetAsync(bb_dev + 3, 0, 4 * sizeof(unsigned long long), ctx->stream));
  bbox_kernel<<<min(blocks(N, 256), 2u * ctx->num_sms), 256, 0, ctx->stream>>>(pts, N, bb_dev);
  CG_LAUNCH_CHECK(ctx);
  unsigned long long bb[7];
  CG_CUDA(ctx, cudaMemcpyAsync(bb, bb_dev, sizeof(bb), cudaMemcpyDeviceToHost, ctx->stream));
  CG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  CG_REQUIRE(ctx, bb[6] == 0, "point coordinates must be finite");
  for (int a = 0; a < 3; a++) { mn[a] = key2d(bb[a]); mx[a] = key2d(bb[3 + a]); }
  return CG_OK;
}

uint32_t table_cap(int n) {
  uint32_t c = 64;
  while (c < 2u * (uint32_t)n) c <<= 1;
  return c;
}

}  // namespace

extern "C" int cg_cloud_create_dev(cg_ctx *ctx, const double *pts, int N, double cell, cg_cloud **out) {
  if (!ctx || !out) return CG_EINVAL;
  *out = nullptr;
  CG_REQUIRE(ctx, N >= 0 && (pts || N == 0), "cloud_create: bad points");
  CG_REQUIRE(ctx, cell > 0.0 && std::isfinite(cell), "cloud_create: cell must be positive and finite");
  CG_REQUIRE(ctx, N < (1 << 30), "cloud_create: at most 2^30 points");
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  cg_cloud *c = new cg_cloud();
  c->ctx = ctx;
  c->N = N;
  c->cell = cell;
  if (N == 0) { *out = c; return CG_OK; }
  int rc = CG_OK;
  auto fail = [&](int code) { cudaFree(c->spts); cudaFree(c->sidx); cudaFree(c->fine); cudaFree(c->coarse); delete c; return code; };

  // temporaries: keys (2 N), values (2 N), run-length outputs, cub scratch -- all from the context arena
  size_t sort_b = 0, rle_b = 0, scan_b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_b, (unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                  (int32_t *)nullptr, (int32_t *)nullptr, N, 0, 63);
  cub::DeviceRunLengthEncode::Encode(nullptr, rle_b, (unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                     (int *)nullptr, (int *)nullptr, N);
  cub::DeviceScan::ExclusiveSum(nullptr, scan_b, (int *)nullptr, (int *)nullptr, N);
  const size_t cub_b = std::max(sort_b, std::max(rle_b, scan_b));
  const size_t ws = cg_arena::pad(8 * sizeof(unsigned long long)) + 3 * cg_arena::pad(N * 8ull) + 4 * cg_arena::pad(N * 4ull) +
                    cg_arena::pad(2 * sizeof(int)) + cg_arena::pad(cub_b);
  if ((rc = cg_ws_reserve(ctx, ws)) != CG_OK) return fail(rc);
  cg_arena ar(ctx->ws);
  auto *bb = ar.take<unsigned long long>(8);
  auto *k0 = ar.take<unsigned long long>(N), *k1 = ar.take<unsigned long long>(N), *uniq = ar.take<unsigned long long>(N);
  auto *v0 = ar.take<int32_t>(N), *v1 = ar.take<int32_t>(N), *cnt = ar.take<int32_t>(N), *st = ar.take<int32_t>(N);
  auto *nruns = ar.take<int>(2);
  void *tmp = ar.take<char>(cub_b);

  if ((rc = device_bbox(ctx, pts, N, bb, c->org, c->bmax)) != CG_OK) return fail(rc);
  for (int a = 0; a < 3; a++) {
    const double span = (c->bmax[a] - c->org[a]) / cell;
    if (!(span < (double)(MAX_AXIS_CELLS - 1))) {
      ctx->err = "invalid argument: cloud_create: cell too small for the cloud's extent (2^21 cells per axis)";
      return fail(CG_EINVAL);
    }
    c->dims[a] = (int)floor(span) + 1;
    c->cdims[a] = ((c->dims[a] - 1) >> CBITS) + 1;
  }
  const int endbit = bits_for((long)coarse_lin(c->cdims, c->cdims[0] - 1, c->cdims[1] - 1, c->cdims[2] - 1)) + 3 * CBITS;
  const Grid g0 = view(c);
  cell_key_kernel<<<blocks(N, 256), 256, 0, ctx->stream>>>(pts, N, g0, k0, v0);
  CG_LAUNCH_CHECK(ctx);
  size_t b = cub_b;
  CG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, b, k0, k1, v0, v1, N, 0, endbit, ctx->stream));
  CG_CUDA(ctx, cudaMalloc(&c->spts, (size_t)N * 3 * sizeof(double)));
  CG_CUDA(ctx, cudaMalloc(&c->sidx, (size_t)N * sizeof(int32_t)));
  gather_kernel<<<blocks(N, 256), 256, 0, ctx->stream>>>(pts, v1, N, c->spts, c->sidx, k1, k0);
  CG_LAUNCH_CHECK(ctx);
  // fine runs of k1 -> (uniq, cnt, st); coarse runs of k0 (= k1 >> 9) follow once the fine table is built
  b = cub_b;
  CG_CUDA(ctx, cub::DeviceRunLengthEncode::Encode(tmp, b, k1, uniq, cnt, nruns, N, ctx->stream));
  b = cub_b;
  CG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, b, cnt, st, N, ctx->stream));
  int nr = 0;
  CG_CUDA(ctx, cudaMemcpyAsync(&nr, nruns, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  uint32_t cap = table_cap(nr);
  CG_CUDA(ctx, cudaMalloc(&c->fine, cap * sizeof(HashE)));
  c->fmask = cap - 1;
  CG_CUDA(ctx, cudaMemsetAsync(c->fine, 0xff, cap * sizeof(HashE), ctx->stream));
  hash_insert_kernel<<<blocks(nr, 256), 256, 0, ctx->stream>>>(uniq, cnt, st, nruns, c->fine, c->fmask);
  CG_LAUNCH_CHECK(ctx);
  b = cub_b;
  CG_CUDA(ctx, cub::DeviceRunLengthEncode::Encode(tmp, b, k0, uniq, cnt, nruns + 1, N, ctx->stream));
  b = cub_b;
  CG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, b, cnt, st, N, ctx->stream));
  CG_CUDA(ctx, cudaMemcpyAsync(&nr, nruns + 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  cap = table_cap(nr);
  CG_CUDA(ctx, cudaMalloc(&c->coarse, cap * sizeof(HashE)));
  c->cmask = cap - 1;
  CG_CUDA(ctx, cudaMemsetAsync(c->coarse, 0xff, cap * sizeof(HashE), ctx->stream));
  hash_insert_kernel<<<blocks(nr, 256), 256, 0, ctx->stream>>>(uniq, cnt, st, nruns + 1, c->coarse, c->cmask);
  CG_LAUNCH_CHECK(ctx);
  *out = c;
  return CG_OK;
}

extern "C" void cg_cloud_destroy(cg_cloud *c) {
  if (!c) return;
  cudaSetDevice(c->ctx->device);
  cudaFree(c->spts);
  cudaFree(c->sidx);
  cudaFree(c->fine);
  cudaFree(c->coarse);
  delete c;
}

extern "C" int cg_cloud_nearest_dev(cg_cloud *c, const double *q, int Q, double *out_dist, int32_t *out_idx) {
  if (!c) return CG_EINVAL;
  cg_ctx *ctx = c->ctx;
  CG_REQUIRE(ctx, Q >= 0 && (Q == 0 || (q && out_dist && out_idx)), "cloud_nearest: bad arguments");
  if (Q == 0) return CG_OK;
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  nearest_kernel<<<blocks(Q, 128), 128, 0, ctx->stream>>>(view(c), q, Q, out_dist, out_idx);
  CG_LAUNCH_CHECK(ctx);
  return CG_OK;
}

extern "C" int cg_cloud_any_within_dev(cg_cloud *c, const double *q, int Q, double r, uint8_t *out) {
  if (!c) return CG_EINVAL;
  cg_ctx *ctx = c->ctx;
  CG_REQUIRE(ctx, Q >= 0 && (Q == 0 || (q && out)), "cloud_any_within: bad arguments");
  CG_REQUIRE(ctx, r >= 0.0 && std::isfinite(r), "cloud_any_within: r must be finite and >= 0");
  if (Q == 0) return CG_OK;
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  any_within_kernel<<<blocks(Q, 128), 128, 0, ctx->stream>>>(view(c), q, Q, r, out);
  CG_LAUNCH_CHECK(ctx);
  return CG_OK;
}

extern "C" int cg_cloud_normals_dev(cg_cloud *c, double radius, int max_nn, const double view_port[3], double *out_nrm,
                                    int32_t *out_nbr) {
  if (!c) return CG_EINVAL;
  cg_ctx *ctx = c->ctx;
  CG_REQUIRE(ctx, radius > 0.0 && std::isfinite(radius), "cloud_normals: radius must be positive and finite");
  CG_REQUIRE(ctx, max_nn >= 1 && max_nn <= 32, "cloud_normals: max_nn must be in [1, 32]");
  CG_REQUIRE(ctx, view_port && std::isfinite(view_port[0]) && std::isfinite(view_port[1]) && std::isfinite(view_port[2]),
             "cloud_normals: view_port must be finite");
  CG_REQUIRE(ctx, out_nrm || c->N == 0, "cloud_normals: bad output");
  const double span = 2.0 * radius / c->cell + 2.0;
  CG_REQUIRE(ctx, span * span * span < (double)(1 << 30), "cloud_normals: radius too large for the index's cell size");
  if (c->N == 0) return CG_OK;
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  normals_kernel<<<blocks(c->N, NW * 32), NW * 32, 0, ctx->stream>>>(view(c), radius, radius * radius, max_nn, view_port[0],
                                                                    view_port[1], view_port[2], out_nrm, out_nbr);
  CG_LAUNCH_CHECK(ctx);
  return CG_OK;
}

extern "C" int cg_voxel_down_sample_dev(cg_ctx *ctx, const double *pts, const double *nrm, int N, double voxel,
                                        double *out_pts, double *out_nrm, int32_t *out_count) {
  if (!ctx) return CG_EINVAL;
  CG_REQUIRE(ctx, N >= 0 && out_count && (N == 0 || (pts && out_pts && (!nrm || out_nrm))), "voxel_down_sample: bad arguments");
  CG_REQUIRE(ctx, voxel > 0.0 && std::isfinite(voxel), "voxel_down_sample: voxel_size must be positive and finite");
  CG_REQUIRE(ctx, N < (1 << 30), "voxel_down_sample: at most 2^30 points");
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  if (N == 0) {
    CG_CUDA(ctx, cudaMemsetAsync(out_count, 0, sizeof(int32_t), ctx->stream));
    return CG_OK;
  }
  size_t sort_b = 0, scan_b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_b, (unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                  (int32_t *)nullptr, (int32_t *)nullptr, N, 0, 64);
  cub::DeviceScan::ExclusiveSum(nullptr, scan_b, (int32_t *)nullptr, (int32_t *)nullptr, N);
  const size_t cub_b = std::max(sort_b, scan_b);
  const size_t ws = cg_arena::pad(8 * sizeof(unsigned long long)) + 2 * cg_arena::pad(N * 8ull) + cg_arena::pad(N * 12ull) +
                    5 * cg_arena::pad(N * 4ull) + cg_arena::pad(cub_b);
  int rc;
  if ((rc = cg_ws_reserve(ctx, ws)) != CG_OK) return rc;
  cg_arena ar(ctx->ws);
  auto *bb = ar.take<unsigned long long>(8);
  auto *k0 = ar.take<unsigned long long>(N), *k1 = ar.take<unsigned long long>(N);
  auto *vi = ar.take<int32_t>(3 * (size_t)N);
  auto *o0 = ar.take<int32_t>(N), *o1 = ar.take<int32_t>(N), *head = ar.take<int32_t>(N), *slot = ar.take<int32_t>(N);
  auto *seg = ar.take<int32_t>(N);
  void *tmp = ar.take<char>(cub_b);

  double mn[3], mx[3];
  if ((rc = device_bbox(ctx, pts, N, bb, mn, mx)) != CG_OK) return rc;
  double vmin[3], vmax[3], span = 0.0;
  for (int a = 0; a < 3; a++) {
    vmin[a] = mn[a] - voxel * 0.5;
    vmax[a] = mx[a] + voxel * 0.5;
    span = std::max(span, vmax[a] - vmin[a]);
  }
  // open3d: "voxel_size is too small" when the index range does not fit an int
  CG_REQUIRE(ctx, !(voxel * (double)INT_MAX < span), "voxel_down_sample: voxel_size is too small (index range beyond int32)");
  int bits[3];
  for (int a = 0; a < 3; a++) bits[a] = bits_for((long)floor((mx[a] - vmin[a]) / voxel));
  voxel_index_kernel<<<blocks(N, 256), 256, 0, ctx->stream>>>(pts, N, vmin[0], vmin[1], vmin[2], voxel, vi, o0);
  CG_LAUNCH_CHECK(ctx);
  // LSD passes of stable radix sorts: pack as many trailing axes into 64 bits as fit, least significant first
  int32_t *ord = o0, *alt = o1;
  for (int a1 = 3; a1 > 0;) {
    int a0 = a1, nb = 0;
    while (a0 > 0 && nb + bits[a0 - 1] <= 64) nb += bits[--a0];
    if (nb > 0) {
      voxel_key_kernel<<<blocks(N, 256), 256, 0, ctx->stream>>>(vi, ord, N, a0, a1, bits[1], bits[2], k0);
      CG_LAUNCH_CHECK(ctx);
      size_t b = cub_b;
      CG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, b, k0, k1, ord, alt, N, 0, nb, ctx->stream));
      std::swap(ord, alt);
    }
    a1 = a0;
  }
  voxel_head_kernel<<<blocks(N, 256), 256, 0, ctx->stream>>>(vi, ord, N, head);
  CG_LAUNCH_CHECK(ctx);
  size_t b = cub_b;
  CG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, b, head, slot, N, ctx->stream));
  voxel_seg_kernel<<<blocks(N, 256), 256, 0, ctx->stream>>>(head, slot, N, seg, out_count);
  CG_LAUNCH_CHECK(ctx);
  voxel_mean_kernel<<<blocks(N, 128), 128, 0, ctx->stream>>>(pts, nrm, ord, seg, out_count, N, out_pts, out_nrm);
  CG_LAUNCH_CHECK(ctx);
  return CG_OK;
}
