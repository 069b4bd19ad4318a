// D1 / D2 geometry sums (myutils/pc_error_wrapper.py geometry_metrics) on the device: exact nearest neighbours through a uniform
// grid, per-point p2point / p2plane values in NumPy's arithmetic, and a fixed-order reduction.  Contract in include/pcgc_b200.h
// (pcgc_geometry_sums).  The same grid and search, widened from one to k nearest neighbours, give the PCA normals of
// pcgc_estimate_normals (knn_normals_kernel).
//
// Grid over a searched set S (n points):
//   - cell size h = the smallest (to 1e-9 relative) for which the dense table has at most kCellsPerPoint * n cells, found by bisection
//     on the device from the bounding box: the table is bounded by the point count for any extent (vox10, vox12, float, negative);
//   - points sorted by linear cell id with a stable radix sort, so the points of a cell are contiguous and in ascending index order;
//     a row of cells along x is one contiguous range of the sorted points;
//   - a coarse occupancy level (kCoarse^3 fine cells per coarse cell) bounds the cost of far queries (Hausdorff outliers): after
//     kFineRings fine rings the search continues ring by ring over the coarse cells and skips the empty ones (and the fine rows
//     already scanned, so that no point is visited twice).
// A query q is first clamped to the bounding box (q'); for every p of S, |q - p|^2 >= |q - q'|^2 + |q' - p|^2, and the points of the
// cells outside a ring of radius r around the cell of q' are at least `lb` from q', lb = distance from q' to that ring's outer faces
// on the sides where the grid continues (less a slack of 1e-12 of the grid's coordinate range for the rounding of the cell index).
// The search stops when (|q - q'|^2 + lb^2) * (1 - 1e-12) > best or no cell is left: exact, nothing capped.
//
// Tie rule: among equidistant neighbours the LOWEST index of the searched array wins ((d2, index) lexicographic minimum).
// Per-point arithmetic: e = q - p, |e|^2 = (e0*e0 + e1*e1) + e2*e2, e.n = (e0*n0 + e1*n1) + e2*n2, squared; this file is built with
// -fmad=false (build.py PER_FILE), so every multiply and add rounds on its own, as in NumPy.
// Reductions: per-query values are stored, then summed in a fixed two-stage order (kRedBlocks contiguous chunks, a fixed shared-memory
// tree in each, one block over the partials).  No floating-point atomics.  For integer coordinates every |e|^2 and every partial sum
// is an integer below 2^53, so the float64 p2point sums are exact and do not depend on the order at all.
#include <cub/cub.cuh>
#include <float.h>
#include <math.h>

#include "common.cuh"

namespace pcgc {

namespace {

constexpr int kCellsPerPoint = 8;   // dense table: at most 8 * n + 8 cells (int32 counts + starts: <= 64 B per searched point)
constexpr int kCoarse = 8;          // fine cells per coarse cell per axis
constexpr int kFineRings = 2;       // fine rings (radius 0..2) before the coarse search
constexpr int kRedBlocks = 512;     // stage-1 blocks of the reduction (fixed: the summation order depends on n only)
constexpr int kThreads = 256;

struct GridParams {
  double lo[3], hi[3];
  double h, hc;        // fine / coarse cell size
  double inv_h;        // 1 / h: the cell index is floor((x - lo) * inv_h) everywhere (a double division is a subroutine call)
  double slack;
  int G[3], Gc[3];
};

struct SortedPoint { double x, y, z, idx; };    // 32 B; idx < 2^31 is exact in a double

struct Grid {
  GridParams* params = nullptr;
  double* partial = nullptr;      // [kRedBlocks][6] bounding-box partials
  uint32_t* keys[2] = {nullptr, nullptr};
  int32_t* vals[2] = {nullptr, nullptr};
  int32_t* counts = nullptr;      // [cells_cap]
  int32_t* starts = nullptr;      // [cells_cap + 1]
  int32_t* coarse = nullptr;      // [cells_cap] occupancy counts of the coarse cells
  SortedPoint* pts = nullptr;     // [n]
  const int32_t* order = nullptr; // sorted indices (points of the set in cell order)
};

__device__ __forceinline__ int cell_of(double x, double lo, double inv_h, int G) {
  const double t = floor((x - lo) * inv_h);
  if (!(t > 0.0)) return 0;
  if (t > (double)(G - 1)) return G - 1;
  return (int)t;
}

__global__ void bbox_partial_kernel(const double* __restrict__ p, int64_t n, double* __restrict__ partial) {
  __shared__ double s[6][kThreads];
  double mn[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, mx[3] = {-DBL_MAX, -DBL_MAX, -DBL_MAX};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    for (int k = 0; k < 3; ++k) { const double v = p[3 * i + k]; mn[k] = fmin(mn[k], v); mx[k] = fmax(mx[k], v); }
  for (int k = 0; k < 3; ++k) { s[k][threadIdx.x] = mn[k]; s[3 + k][threadIdx.x] = mx[k]; }
  __syncthreads();
  for (int w = kThreads / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w)
      for (int k = 0; k < 3; ++k) {
        s[k][threadIdx.x] = fmin(s[k][threadIdx.x], s[k][threadIdx.x + w]);
        s[3 + k][threadIdx.x] = fmax(s[3 + k][threadIdx.x], s[3 + k][threadIdx.x + w]);
      }
    __syncthreads();
  }
  if (threadIdx.x < 6) partial[blockIdx.x * 6 + threadIdx.x] = s[threadIdx.x][0];
}

__device__ __forceinline__ double grid_cells(const double* e, double h) {
  double c = 1.0;
  for (int k = 0; k < 3; ++k) c *= floor(e[k] / h) + 1.0;
  return c;
}

// One thread: bounding box from the partials, then the cell size by bisection.
__global__ void grid_params_kernel(const double* __restrict__ partial, int nb, int64_t n, GridParams* __restrict__ gp) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  GridParams g;
  for (int k = 0; k < 3; ++k) { g.lo[k] = DBL_MAX; g.hi[k] = -DBL_MAX; }
  for (int b = 0; b < nb; ++b)
    for (int k = 0; k < 3; ++k) { g.lo[k] = fmin(g.lo[k], partial[b * 6 + k]); g.hi[k] = fmax(g.hi[k], partial[b * 6 + 3 + k]); }
  double e[3], emax = 0.0, amax = 0.0;
  for (int k = 0; k < 3; ++k) {
    e[k] = g.hi[k] - g.lo[k];
    emax = fmax(emax, e[k]);
    amax = fmax(amax, fmax(fabs(g.lo[k]), fabs(g.hi[k])));
  }
  const double cap = (double)kCellsPerPoint * (double)n;
  double h;
  if (emax == 0.0) {
    h = 1.0;                                     // one point, or all points equal: one cell
  } else {
    double hi_h = emax, lo_h = emax * 1e-12;     // grid_cells(hi_h) <= 8 <= cap; bisection keeps grid_cells(hi_h) <= cap
    if (grid_cells(e, lo_h) <= cap) hi_h = lo_h;
    else
      for (int it = 0; it < 200 && hi_h - lo_h > 1e-9 * hi_h; ++it) {
        const double mid = 0.5 * (lo_h + hi_h);
        if (grid_cells(e, mid) <= cap) hi_h = mid; else lo_h = mid;
      }
    h = hi_h;
  }
  g.h = h;
  g.hc = h * kCoarse;
  g.inv_h = 1.0 / h;
  for (int k = 0; k < 3; ++k) {
    g.G[k] = (int)(floor(e[k] / h) + 1.0);
    g.Gc[k] = (g.G[k] + kCoarse - 1) / kCoarse;
  }
  g.slack = 1e-12 * (amax + emax + g.hc);
  *gp = g;
}

__global__ void cell_key_kernel(const double* __restrict__ p, int64_t n, const GridParams* __restrict__ gp, uint32_t* __restrict__ keys,
                                int32_t* __restrict__ vals, int32_t* __restrict__ counts, int32_t* __restrict__ coarse) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const GridParams& g = *gp;
  int c[3];
  for (int k = 0; k < 3; ++k) c[k] = cell_of(p[3 * i + k], g.lo[k], g.inv_h, g.G[k]);
  const uint32_t id = (uint32_t)(((int64_t)c[2] * g.G[1] + c[1]) * g.G[0] + c[0]);
  keys[i] = id;
  vals[i] = (int32_t)i;
  atomicAdd(&counts[id], 1);                    // integer counts: the result does not depend on the order
  const int64_t cid = ((int64_t)(c[2] / kCoarse) * g.Gc[1] + c[1] / kCoarse) * g.Gc[0] + c[0] / kCoarse;
  atomicAdd(&coarse[cid], 1);
}

__global__ void gather_sorted_kernel(const double* __restrict__ p, int64_t n, const int32_t* __restrict__ order, SortedPoint* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int32_t i = order[j];
  out[j] = SortedPoint{p[3 * i], p[3 * i + 1], p[3 * i + 2], (double)i};
}

struct Best {
  double d2 = DBL_MAX;
  int idx = 0x7fffffff;
};

__device__ __forceinline__ void scan_range(const SortedPoint* __restrict__ pts, int j0, int j1, double q0, double q1, double q2, Best& b) {
  for (int j = j0; j < j1; ++j) {
    const SortedPoint p = pts[j];
    const double e0 = q0 - p.x, e1 = q1 - p.y, e2 = q2 - p.z;
    const double d2 = (e0 * e0 + e1 * e1) + e2 * e2;
    const int idx = (int)p.idx;
    if (d2 < b.d2 || (d2 == b.d2 && idx < b.idx)) { b.d2 = d2; b.idx = idx; }
  }
}

// Distance from qc to the outside of the box of cells [c - r, c + r] on the sides where the grid (dims G, cell size s) continues;
// DBL_MAX when no cell is left outside.
__device__ __forceinline__ double outside_distance(const GridParams& g, const double* qc, const int* c, int r, double s, const int* G) {
  double lb = DBL_MAX;
  for (int k = 0; k < 3; ++k) {
    if (c[k] - r > 0) lb = fmin(lb, qc[k] - (g.lo[k] + (double)(c[k] - r) * s));
    if (c[k] + r < G[k] - 1) lb = fmin(lb, (g.lo[k] + (double)(c[k] + r + 1) * s) - qc[k]);
  }
  return lb;
}

__device__ __forceinline__ bool done_after(const GridParams& g, double lb, double dq2, double best) {
  if (lb == DBL_MAX) return true;
  lb = fmax(lb - g.slack, 0.0);
  return (dq2 + lb * lb) * (1.0 - 1e-12) > best;
}

// The exact search around the query qc (clamped to the bounding box, |q - qc|^2 = dq2) in cell c: every fine ring r = 0..kFineRings,
// then every coarse ring over the occupied coarse cells, skipping the fine rows already scanned, so that every point is visited at most
// once.  scan(j0, j1) visits the sorted points [j0, j1); the walk ends when done_after holds for bound() (the d2 an unvisited point
// must beat) or no cell is left.
template <class Scan, class Bound>
__device__ __forceinline__ void ring_search(const GridParams& g, const int32_t* __restrict__ starts, const int32_t* __restrict__ coarse,
                                            const double* qc, const int* c, double dq2, Scan&& scan, Bound&& bound) {
  const int Gx = g.G[0], Gy = g.G[1];
  bool done = false;
  for (int r = 0; r <= kFineRings && !done; ++r) {
    for (int z = max(c[2] - r, 0); z <= min(c[2] + r, g.G[2] - 1); ++z)
      for (int y = max(c[1] - r, 0); y <= min(c[1] + r, Gy - 1); ++y) {
        const int64_t base = ((int64_t)z * Gy + y) * Gx;
        if (abs(z - c[2]) == r || abs(y - c[1]) == r) {
          const int x0 = max(c[0] - r, 0), x1 = min(c[0] + r, Gx - 1);
          scan(starts[base + x0], starts[base + x1 + 1]);
        } else {
          if (c[0] - r >= 0) scan(starts[base + c[0] - r], starts[base + c[0] - r + 1]);
          if (c[0] + r < Gx) scan(starts[base + c[0] + r], starts[base + c[0] + r + 1]);
        }
      }
    done = done_after(g, outside_distance(g, qc, c, r, g.h, g.G), dq2, bound());
  }
  if (done) return;
  const int R = kFineRings;
  const int cc[3] = {c[0] / kCoarse, c[1] / kCoarse, c[2] / kCoarse};
  const int Cx = g.Gc[0], Cy = g.Gc[1], Cz = g.Gc[2];
  for (int r = 0; !done; ++r) {
    for (int z = max(cc[2] - r, 0); z <= min(cc[2] + r, Cz - 1); ++z)
      for (int y = max(cc[1] - r, 0); y <= min(cc[1] + r, Cy - 1); ++y) {
        const bool full = abs(z - cc[2]) == r || abs(y - cc[1]) == r;
        const int xa = max(cc[0] - r, 0), xb = min(cc[0] + r, Cx - 1);
        for (int x = xa; x <= xb; ++x) {
          if (!full && x != cc[0] - r && x != cc[0] + r) continue;     // inner rows: only the two end cells are on the ring
          if (coarse[((int64_t)z * Cy + y) * Cx + x] == 0) continue;
          const int fx0 = x * kCoarse, fx1 = min(fx0 + kCoarse, Gx) - 1;
          for (int fz = z * kCoarse; fz < min(z * kCoarse + kCoarse, g.G[2]); ++fz)
            for (int fy = y * kCoarse; fy < min(y * kCoarse + kCoarse, Gy); ++fy) {
              const int64_t base = ((int64_t)fz * Gy + fy) * Gx;
              if (abs(fz - c[2]) <= R && abs(fy - c[1]) <= R) {            // a row through the fine box: only the cells outside it
                const int l1 = min(fx1, c[0] - R - 1), r0 = max(fx0, c[0] + R + 1);
                if (fx0 <= l1) scan(starts[base + fx0], starts[base + l1 + 1]);
                if (r0 <= fx1) scan(starts[base + r0], starts[base + fx1 + 1]);
              } else {
                scan(starts[base + fx0], starts[base + fx1 + 1]);
              }
            }
        }
      }
    done = done_after(g, outside_distance(g, qc, cc, r, g.hc, g.Gc), dq2, bound());
  }
}

// One thread per query.  Queries come in the cell order of their own set (neighbouring threads search neighbouring cells).
// dir 1: normal of the query (normals[qi]); dir 2: normal of the neighbour found (normals[bi]).
__global__ void __launch_bounds__(kThreads, 3) query_kernel(const SortedPoint* __restrict__ queries, int64_t nq, const GridParams* __restrict__ gp,
                                                         const int32_t* __restrict__ starts, const int32_t* __restrict__ coarse,
                                                         const SortedPoint* __restrict__ pts, const double* __restrict__ searched,
                                                         const double* __restrict__ normals, int dir, double* __restrict__ pp,
                                                         double* __restrict__ pl) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nq) return;
  const GridParams g = *gp;
  const SortedPoint qp = queries[t];
  const double q[3] = {qp.x, qp.y, qp.z};
  const int qi = (int)qp.idx;
  double qc[3], dq2 = 0.0;
  int c[3];
  for (int k = 0; k < 3; ++k) {
    qc[k] = fmin(fmax(q[k], g.lo[k]), g.hi[k]);
    const double d = q[k] - qc[k];
    dq2 = dq2 + d * d;
    c[k] = cell_of(qc[k], g.lo[k], g.inv_h, g.G[k]);
  }
  Best b;
  ring_search(g, starts, coarse, qc, c, dq2, [&](int j0, int j1) { scan_range(pts, j0, j1, q[0], q[1], q[2], b); },
              [&]() { return b.d2; });
  const double* p = searched + 3 * (int64_t)b.idx;
  const double e0 = q[0] - p[0], e1 = q[1] - p[1], e2 = q[2] - p[2];
  pp[qi] = (e0 * e0 + e1 * e1) + e2 * e2;
  if (normals) {
    const double* nn = normals + 3 * (int64_t)(dir == 1 ? qi : b.idx);
    const double en = (e0 * nn[0] + e1 * nn[1]) + e2 * nn[2];
    pl[qi] = en * en;
  }
}

// ---- k nearest neighbours and PCA normals (pcgc_estimate_normals) -------------------------------------------------------------------
// One thread per query, queries in the cell order of the set.  The k best (d2, index) pairs are kept sorted in a per-thread array of
// CAP slots (CAP = 16, 32 or 64 >= k): local memory, since it is indexed dynamically.
template <int CAP>
struct KBest {
  double d2[CAP];
  int idx[CAP];
  int count = 0;       // slots held (<= kk)
  int kk;              // min(k, n)
  __device__ __forceinline__ double kth() const { return count >= kk ? d2[kk - 1] : DBL_MAX; }
};

template <int CAP>
__device__ __forceinline__ void knn_scan(const SortedPoint* __restrict__ pts, int j0, int j1, const double* q, KBest<CAP>& b) {
  for (int j = j0; j < j1; ++j) {
    const SortedPoint p = pts[j];
    const double e0 = q[0] - p.x, e1 = q[1] - p.y, e2 = q[2] - p.z;
    const double d2 = (e0 * e0 + e1 * e1) + e2 * e2;
    const int idx = (int)p.idx;
    if (b.count == b.kk) {
      const double w = b.d2[b.kk - 1];
      if (!(d2 < w || (d2 == w && idx < b.idx[b.kk - 1]))) continue;
    }
    int pos = b.count < b.kk ? b.count : b.kk - 1;
    while (pos > 0 && (d2 < b.d2[pos - 1] || (d2 == b.d2[pos - 1] && idx < b.idx[pos - 1]))) {
      b.d2[pos] = b.d2[pos - 1]; b.idx[pos] = b.idx[pos - 1]; --pos;
    }
    b.d2[pos] = d2; b.idx[pos] = idx;
    if (b.count < b.kk) ++b.count;
  }
}

// Cyclic Jacobi on the symmetric 3x3 matrix A (overwritten), at most kJacobiSweeps sweeps; returns the unit eigenvector of
// the smallest eigenvalue (lowest axis on an exact tie of eigenvalues) with the sign rule of the header.
constexpr int kJacobiSweeps = 32;

__device__ void smallest_eigenvector(double A[3][3], double* out) {
  double V[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}};
  const int P[3] = {0, 0, 1}, Q[3] = {1, 2, 2};
  for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
    if (A[0][1] == 0.0 && A[0][2] == 0.0 && A[1][2] == 0.0) break;
    for (int r = 0; r < 3; ++r) {
      const int p = P[r], q = Q[r], o = 3 - p - q;
      const double apq = A[p][q];
      if (apq == 0.0) continue;
      const double g = 100.0 * fabs(apq);
      if (sweep > 3 && fabs(A[p][p]) + g == fabs(A[p][p]) && fabs(A[q][q]) + g == fabs(A[q][q])) {
        A[p][q] = A[q][p] = 0.0;                     // below the rounding of both diagonal entries
        continue;
      }
      const double h = A[q][q] - A[p][p];
      double t;
      if (fabs(h) + g == fabs(h)) {
        t = apq / h;
      } else {
        const double theta = 0.5 * h / apq;
        t = 1.0 / (fabs(theta) + sqrt(1.0 + theta * theta));
        if (theta < 0.0) t = -t;
      }
      const double c = 1.0 / sqrt(1.0 + t * t), sn = t * c, tau = sn / (1.0 + c);
      A[p][p] = A[p][p] - t * apq;
      A[q][q] = A[q][q] + t * apq;
      A[p][q] = A[q][p] = 0.0;
      const double gp = A[o][p], gq = A[o][q];
      A[o][p] = A[p][o] = gp - sn * (gq + gp * tau);
      A[o][q] = A[q][o] = gq + sn * (gp - gq * tau);
      for (int i = 0; i < 3; ++i) {
        const double vp = V[i][p], vq = V[i][q];
        V[i][p] = vp - sn * (vq + vp * tau);
        V[i][q] = vq + sn * (vp - vq * tau);
      }
    }
  }
  int m = 0;
  for (int i = 1; i < 3; ++i)
    if (A[i][i] < A[m][m]) m = i;
  double v[3] = {V[0][m], V[1][m], V[2][m]};
  const double inv = 1.0 / sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
  int a = 0;
  for (int i = 0; i < 3; ++i) {
    v[i] = v[i] * inv;
    if (fabs(v[i]) > fabs(v[a])) a = i;
  }
  const double sg = v[a] < 0.0 ? -1.0 : 1.0;
  for (int i = 0; i < 3; ++i) out[i] = v[i] * sg + 0.0;     // + 0.0: no negative zeros
}

template <int CAP>
__global__ void __launch_bounds__(kThreads) knn_normals_kernel(const SortedPoint* __restrict__ pts, int64_t n, int k,
                                                               const GridParams* __restrict__ gp, const int32_t* __restrict__ starts,
                                                               const int32_t* __restrict__ coarse, const double* __restrict__ src,
                                                               double* __restrict__ normals, int32_t* __restrict__ knn) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const GridParams g = *gp;
  const SortedPoint qp = pts[t];
  const double q[3] = {qp.x, qp.y, qp.z};      // a point of the set: inside the bounding box, so no clamping
  const int qi = (int)qp.idx;
  int c[3];
  for (int d = 0; d < 3; ++d) c[d] = cell_of(q[d], g.lo[d], g.inv_h, g.G[d]);
  KBest<CAP> b;
  b.kk = (int)min((int64_t)k, n);
  ring_search(g, starts, coarse, q, c, 0.0, [&](int j0, int j1) { knn_scan(pts, j0, j1, q, b); }, [&]() { return b.kth(); });
  const int m = b.count;
  if (knn)
    for (int j = 0; j < k; ++j) knn[(int64_t)qi * k + j] = j < m ? b.idx[j] : -1;
  // Covariance about the centroid, in coordinates relative to the query (u = p - q): two passes in (d2, index) order.
  double mu[3] = {0.0, 0.0, 0.0};
  for (int j = 0; j < m; ++j) {
    const double* p = src + 3 * (int64_t)b.idx[j];
    for (int d = 0; d < 3; ++d) mu[d] = mu[d] + (p[d] - q[d]);
  }
  for (int d = 0; d < 3; ++d) mu[d] = mu[d] / (double)m;
  double C[3][3] = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
  for (int j = 0; j < m; ++j) {
    const double* p = src + 3 * (int64_t)b.idx[j];
    const double e[3] = {(p[0] - q[0]) - mu[0], (p[1] - q[1]) - mu[1], (p[2] - q[2]) - mu[2]};
    for (int u = 0; u < 3; ++u)
      for (int v = u; v < 3; ++v) C[u][v] = C[u][v] + e[u] * e[v];
  }
  for (int u = 0; u < 3; ++u)
    for (int v = u; v < 3; ++v) C[v][u] = C[u][v] = C[u][v] / (double)m;
  double nrm[3] = {0.0, 0.0, 1.0};
  if (C[0][0] != 0.0 || C[0][1] != 0.0 || C[0][2] != 0.0 || C[1][1] != 0.0 || C[1][2] != 0.0 || C[2][2] != 0.0)
    smallest_eigenvector(C, nrm);
  for (int d = 0; d < 3; ++d) normals[3 * (int64_t)qi + d] = nrm[d];
}

// Stage 1: block b sums / maxes the contiguous chunk b of the n values of each of `nv` arrays (fixed tree); stage 2 folds the
// kRedBlocks partials the same way.  partial: [nv][kRedBlocks][2].
__global__ void __launch_bounds__(kThreads) reduce_stage1_kernel(const double* __restrict__ v0, const double* __restrict__ v1, int nv,
                                                                 int64_t n, double* __restrict__ partial) {
  __shared__ double ss[kThreads], sm[kThreads];
  const int64_t chunk = (n + kRedBlocks - 1) / kRedBlocks;
  const int64_t a = (int64_t)blockIdx.x * chunk, e = min(a + chunk, n);
  for (int w = 0; w < nv; ++w) {
    const double* v = w == 0 ? v0 : v1;
    double s = 0.0, m = 0.0;
    for (int64_t i = a + threadIdx.x; i < e; i += kThreads) { s = s + v[i]; m = fmax(m, v[i]); }
    ss[threadIdx.x] = s; sm[threadIdx.x] = m;
    __syncthreads();
    for (int k = kThreads / 2; k > 0; k >>= 1) {
      if (threadIdx.x < k) { ss[threadIdx.x] = ss[threadIdx.x] + ss[threadIdx.x + k]; sm[threadIdx.x] = fmax(sm[threadIdx.x], sm[threadIdx.x + k]); }
      __syncthreads();
    }
    if (threadIdx.x == 0) { partial[((int64_t)w * kRedBlocks + blockIdx.x) * 2] = ss[0]; partial[((int64_t)w * kRedBlocks + blockIdx.x) * 2 + 1] = sm[0]; }
    __syncthreads();
  }
}

// out layout [dir][kind][sum, max]; this call writes kinds 0..nv-1 of direction `dir` (0-based).
__global__ void __launch_bounds__(kThreads) reduce_stage2_kernel(const double* __restrict__ partial, int nv, int dir, double* __restrict__ out) {
  __shared__ double ss[kThreads], sm[kThreads];
  for (int w = 0; w < 2; ++w) {
    double s = 0.0, m = 0.0;
    if (w < nv)
      for (int i = threadIdx.x; i < kRedBlocks; i += kThreads) {
        s = s + partial[((int64_t)w * kRedBlocks + i) * 2];
        m = fmax(m, partial[((int64_t)w * kRedBlocks + i) * 2 + 1]);
      }
    ss[threadIdx.x] = s; sm[threadIdx.x] = m;
    __syncthreads();
    for (int k = kThreads / 2; k > 0; k >>= 1) {
      if (threadIdx.x < k) { ss[threadIdx.x] = ss[threadIdx.x] + ss[threadIdx.x + k]; sm[threadIdx.x] = fmax(sm[threadIdx.x], sm[threadIdx.x + k]); }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      out[dir * 4 + w * 2] = w < nv ? ss[0] : 0.0;
      out[dir * 4 + w * 2 + 1] = w < nv ? sm[0] : 0.0;
    }
    __syncthreads();
  }
}

inline unsigned blocks_for(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

}  // namespace

namespace {

// Carves the buffers of one call out of one allocation (256-byte aligned pieces); with base == nullptr it only measures.
struct Carver {
  char* base;
  size_t off = 0;
  template <typename T> T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

struct Plan {
  int64_t n[2] = {0, 0};
  Grid g[2];
  double* pp[2] = {nullptr, nullptr};
  double* pl[2] = {nullptr, nullptr};
  double* red = nullptr;
  void* tmp = nullptr;
  size_t sort_bytes = 0, scan_bytes = 0;
};

void carve_grid(Carver& c, Grid& g, int64_t n) {
  const size_t cells = (size_t)kCellsPerPoint * n + 8;
  g.params = c.take<GridParams>(1);
  g.partial = c.take<double>(kRedBlocks * 6);
  for (int k = 0; k < 2; ++k) { g.keys[k] = c.take<uint32_t>(n); g.vals[k] = c.take<int32_t>(n); }
  g.counts = c.take<int32_t>(cells);
  g.starts = c.take<int32_t>(cells + 1);
  g.coarse = c.take<int32_t>(cells);
  g.pts = c.take<SortedPoint>(n);
}

size_t carve(char* base, Plan& p) {
  Carver c{base};
  for (int s = 0; s < 2; ++s) {
    carve_grid(c, p.g[s], p.n[s]);
    p.pp[s] = c.take<double>(p.n[s]);
    p.pl[s] = c.take<double>(p.n[s]);
  }
  p.red = c.take<double>(2 * kRedBlocks * 2);
  p.tmp = c.take<char>(std::max(p.sort_bytes, p.scan_bytes));
  return c.off + 256;
}

// The normals use one grid (p.g[0] over p.n[0] points) and the sort / scan scratch.
size_t carve_normals(char* base, Plan& p) {
  Carver c{base};
  carve_grid(c, p.g[0], p.n[0]);
  p.tmp = c.take<char>(std::max(p.sort_bytes, p.scan_bytes));
  return c.off + 256;
}

#define GK(call)                            \
  do {                                      \
    cudaError_t e_ = (call);                \
    if (e_ != cudaSuccess) return e_;       \
  } while (0)

cudaError_t build_grid(const double* p, int64_t n, Grid& g, Plan& pl, cudaStream_t s, int64_t* launches) {
  const size_t cells = (size_t)kCellsPerPoint * n + 8;
  bbox_partial_kernel<<<kRedBlocks, kThreads, 0, s>>>(p, n, g.partial);
  grid_params_kernel<<<1, 32, 0, s>>>(g.partial, kRedBlocks, n, g.params);
  GK(cudaMemsetAsync(g.counts, 0, sizeof(int32_t) * cells, s));
  GK(cudaMemsetAsync(g.coarse, 0, sizeof(int32_t) * cells, s));
  cell_key_kernel<<<blocks_for(n), kThreads, 0, s>>>(p, n, g.params, g.keys[0], g.vals[0], g.counts, g.coarse);
  int end_bit = 1;
  while (end_bit < 32 && ((size_t)1 << end_bit) < cells) ++end_bit;
  cub::DoubleBuffer<uint32_t> k(g.keys[0], g.keys[1]);
  cub::DoubleBuffer<int32_t> v(g.vals[0], g.vals[1]);
  size_t bytes = pl.sort_bytes;
  GK(cub::DeviceRadixSort::SortPairs(pl.tmp, bytes, k, v, (int)n, 0, end_bit, s));
  g.order = v.Current();
  bytes = pl.scan_bytes;
  GK(cub::DeviceScan::ExclusiveSum(pl.tmp, bytes, g.counts, g.starts, (int)(cells + 1), s));
  gather_sorted_kernel<<<blocks_for(n), kThreads, 0, s>>>(p, n, g.order, g.pts);
  *launches += 6;      // four kernels; the radix sort and the scan counted as one launch group each
  return cudaGetLastError();
}

}  // namespace

struct GeoWorkspace {
  void* mem = nullptr;
  size_t cap = 0;
  Plan plan;
};

void free_geometry_workspace(GeoWorkspace* ws) {
  if (!ws) return;
  if (ws->mem) cudaFree(ws->mem);
  delete ws;
}

namespace {

// CUB scratch sizes for grids of up to nmax points.
cudaError_t size_scratch(Plan& plan, int64_t nmax, cudaStream_t s) {
  const size_t cells_max = (size_t)kCellsPerPoint * nmax + 8;
  cub::DoubleBuffer<uint32_t> k(nullptr, nullptr);
  cub::DoubleBuffer<int32_t> v(nullptr, nullptr);
  GK(cub::DeviceRadixSort::SortPairs(nullptr, plan.sort_bytes, k, v, (int)nmax, 0, 32, s));
  GK(cub::DeviceScan::ExclusiveSum(nullptr, plan.scan_bytes, (int32_t*)nullptr, (int32_t*)nullptr, (int)(cells_max + 1), s));
  return cudaSuccess;
}

// Grows the workspace to `need` bytes (synchronises only then); *base = its 256-byte aligned start.
cudaError_t reserve(GeoWorkspace** wsp, size_t need, cudaStream_t s, char** base) {
  if (!*wsp) *wsp = new GeoWorkspace();
  GeoWorkspace* ws = *wsp;
  if (ws->cap < need) {
    if (ws->mem) { GK(cudaStreamSynchronize(s)); GK(cudaFree(ws->mem)); ws->mem = nullptr; ws->cap = 0; }
    const size_t want = need + need / 4;
    GK(cudaMalloc(&ws->mem, want));
    ws->cap = want;
  }
  *base = reinterpret_cast<char*>(((uintptr_t)ws->mem + 255) & ~(uintptr_t)255);
  return cudaSuccess;
}

}  // namespace

cudaError_t launch_geometry_grids(GeoWorkspace** wsp, const double* a, int64_t na, const double* b, int64_t nb, cudaStream_t s,
                                  int64_t* launches) {
  Plan plan;
  plan.n[0] = na; plan.n[1] = nb;
  GK(size_scratch(plan, std::max(na, nb), s));
  char* base = nullptr;
  GK(reserve(wsp, carve(nullptr, plan), s, &base));
  GeoWorkspace* ws = *wsp;
  carve(base, plan);
  const double* set[2] = {a, b};
  for (int k = 0; k < 2; ++k) GK(build_grid(set[k], plan.n[k], plan.g[k], plan, s, launches));
  ws->plan = plan;
  return cudaSuccess;
}

cudaError_t launch_geometry_queries(GeoWorkspace* ws, const double* a, const double* b, const double* normals_a, double* out, cudaStream_t s,
                                    int64_t* launches) {
  const Plan& plan = ws->plan;
  const double* set[2] = {a, b};
  // direction 1: A against the grid of B; direction 2: B against the grid of A
  for (int d = 0; d < 2; ++d) {
    const int q = d, t = 1 - d;
    query_kernel<<<blocks_for(plan.n[q]), kThreads, 0, s>>>(plan.g[q].pts, plan.n[q], plan.g[t].params, plan.g[t].starts, plan.g[t].coarse,
                                                            plan.g[t].pts, set[t], normals_a, d + 1, plan.pp[q], plan.pl[q]);
    const int nv = normals_a ? 2 : 1;
    reduce_stage1_kernel<<<kRedBlocks, kThreads, 0, s>>>(plan.pp[q], plan.pl[q], nv, plan.n[q], plan.red);
    reduce_stage2_kernel<<<1, kThreads, 0, s>>>(plan.red, nv, d, out);
    *launches += 3;
  }
  return cudaGetLastError();
}

cudaError_t launch_normals_grid(GeoWorkspace** wsp, const double* p, int64_t n, cudaStream_t s, int64_t* launches) {
  Plan plan;
  plan.n[0] = n;
  GK(size_scratch(plan, n, s));
  char* base = nullptr;
  GK(reserve(wsp, carve_normals(nullptr, plan), s, &base));
  carve_normals(base, plan);
  GK(build_grid(p, n, plan.g[0], plan, s, launches));
  (*wsp)->plan = plan;
  return cudaSuccess;
}

cudaError_t launch_normals_query(GeoWorkspace* ws, const double* p, int64_t n, int k, double* normals, int32_t* knn, cudaStream_t s,
                                 int64_t* launches) {
  const Grid& g = ws->plan.g[0];
  if (k <= 16)
    knn_normals_kernel<16><<<blocks_for(n), kThreads, 0, s>>>(g.pts, n, k, g.params, g.starts, g.coarse, p, normals, knn);
  else if (k <= 32)
    knn_normals_kernel<32><<<blocks_for(n), kThreads, 0, s>>>(g.pts, n, k, g.params, g.starts, g.coarse, p, normals, knn);
  else
    knn_normals_kernel<64><<<blocks_for(n), kThreads, 0, s>>>(g.pts, n, k, g.params, g.starts, g.coarse, p, normals, knn);
  *launches += 1;
  return cudaGetLastError();
}

}  // namespace pcgc
