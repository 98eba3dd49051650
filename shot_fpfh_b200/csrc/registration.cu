// Registration stages downstream of the matcher (SURVEY.md §8f row 4), the data-parallel part of each:
//   RANSAC  (matching/ransac.py:17-82)  the n_draws x n_matches inlier count — the draws replay NumPy's generator on
//           the host and the 4-point Kabsch fits are a batched host SVD; what costs is the count (:55-62).
//   ICP     (icp.py:137-189, core/solvers.py:34-48)  per iteration: transform the subsampled scan, nearest reference
//           point within d_max of each (KDTree.query + the `<= d_max` filter), and the sums of the point-to-plane
//           normal equations g^T g, g^T h plus the residual — one kernel, one 29-double result per iteration.
#include <algorithm>

#include "sf_common.cuh"

namespace sf {

// ---- RANSAC: inliers of every candidate transform ------------------------------------------------------------
// One block per draw. transforms[d] = {R row-major (9), t (3)}; a point is an inlier when
// || R a + t - b || <= threshold (ransac.py:55-62; np.linalg.norm, i.e. the sqrt is taken before comparing).
__global__ void __launch_bounds__(256)
    ransac_inliers_kernel(const double* __restrict__ a, const double* __restrict__ b, int64_t m,
                          const double* __restrict__ transforms, double threshold, int32_t* __restrict__ counts) {
  __shared__ int warp_counts[8];
  const double* tr = transforms + 12 * int64_t(blockIdx.x);
  double r[9], t[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) r[k] = __ldg(tr + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) t[k] = __ldg(tr + 9 + k);
  int count = 0;
  for (int64_t i = threadIdx.x; i < m; i += blockDim.x) {
    const double ax = __ldg(a + 3 * i), ay = __ldg(a + 3 * i + 1), az = __ldg(a + 3 * i + 2);
    const double dx = (r[0] * ax + r[1] * ay + r[2] * az + t[0]) - __ldg(b + 3 * i);
    const double dy = (r[3] * ax + r[4] * ay + r[5] * az + t[1]) - __ldg(b + 3 * i + 1);
    const double dz = (r[6] * ax + r[7] * ay + r[8] * az + t[2]) - __ldg(b + 3 * i + 2);
    count += sqrt(dx * dx + dy * dy + dz * dz) <= threshold;
  }
  count = warp_sum(count);
  if ((threadIdx.x & 31) == 0) warp_counts[threadIdx.x >> 5] = count;
  __syncthreads();
  if (threadIdx.x == 0) {
    int total = 0;
    for (int w = 0; w < int(blockDim.x >> 5); ++w) total += warp_counts[w];
    counts[blockIdx.x] = total;
  }
}

// ---- ICP, point to plane: one iteration's normal equations ---------------------------------------------------
// Per inlier (p = transformed scan point, q = its nearest reference point, n = q's normal):
//   g = [p x n, n] (6), h = (q - p) . n          (solvers.py:39-44)
//   sums: g_i g_j for i <= j (21), g_i h (6), |(p - q) . n| (1, icp.py:176-182), 1 (the inlier count)
constexpr int kIcpTerms = 29;

__device__ __forceinline__ double icp_term(int lane, const double g[6], double h, double residual) {
  // lanes 0..20: the upper triangle of g g^T in row order; 21..26: g h; 27: |residual|; 28: 1
  if (lane < 21) {
    int i = 0, first = 0;
    while (lane >= first + (6 - i)) { first += 6 - i; ++i; }
    const int j = i + (lane - first);
    double gi = g[0], gj = g[0];
#pragma unroll
    for (int k = 1; k < 6; ++k) {
      gi = i == k ? g[k] : gi;
      gj = j == k ? g[k] : gj;
    }
    return gi * gj;
  }
  if (lane < 27) {
    double gi = g[0];
#pragma unroll
    for (int k = 1; k < 6; ++k) gi = (lane - 21) == k ? g[k] : gi;
    return gi * h;
  }
  return lane == 27 ? fabs(residual) : 1.0;
}

// One warp per scan point (grid-stride, so that the order of a warp's additions is fixed by the launch shape):
// the 27 cells around the transformed point are scanned for the nearest reference point; ties go to the lowest
// cell-sorted position. Lane l < 29 accumulates term l; the warp's sums go to partial[warp][29].
__global__ void __launch_bounds__(256)
    icp_plane_kernel(GridView g, const double* __restrict__ scan, int64_t n_scan, const double* __restrict__ transform,
                     double d_max, double* __restrict__ partial, int32_t* __restrict__ nearest) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  const int64_t warps_total = (int64_t(gridDim.x) * blockDim.x) >> 5;
  double r[9], t[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) r[k] = __ldg(transform + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) t[k] = __ldg(transform + 9 + k);
  double acc = 0.0;
  for (int64_t i = warp; i < n_scan; i += warps_total) {
    const double sx = __ldg(scan + 3 * i), sy = __ldg(scan + 3 * i + 1), sz = __ldg(scan + 3 * i + 2);
    const double px = r[0] * sx + r[1] * sy + r[2] * sz + t[0];
    const double py = r[3] * sx + r[4] * sy + r[5] * sz + t[1];
    const double pz = r[6] * sx + r[7] * sy + r[8] * sz + t[2];
    const Runs runs = build_runs(g, px, py, pz, lane);
    const int total = runs.pref[9];
    double best = INFINITY;
    int best_pos = 0x7fffffff;
    for (int v = lane; v < total; v += 32) {
      const int pos = run_position(runs, v);
      const double4 q = load_pt(g.pts + pos);
      const double d2 = rdist3(px - q.x, py - q.y, pz - q.z);
      if (d2 < best || (d2 == best && pos < best_pos)) { best = d2; best_pos = pos; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(kFull, best, o);
      const int op = __shfl_xor_sync(kFull, best_pos, o);
      if (ob < best || (ob == best && op < best_pos)) { best = ob; best_pos = op; }
    }
    const bool inlier = total > 0 && sqrt(best) <= d_max;  // KDTree.query's distance is sqrt(rdist); icp.py:160
    if (nearest != nullptr && lane == 0)
      nearest[i] = inlier ? int32_t(__double_as_longlong(load_pt(g.pts + best_pos).w)) : -1;
    if (inlier) {
      const double4 q = load_pt(g.pts + best_pos), n = load_pt(g.nrm + best_pos);
      const double gv[6] = {py * n.z - pz * n.y, pz * n.x - px * n.z, px * n.y - py * n.x, n.x, n.y, n.z};
      const double h = (q.x - px) * n.x + (q.y - py) * n.y + (q.z - pz) * n.z;
      if (lane < kIcpTerms) acc += icp_term(lane, gv, h, -h);
    }
  }
  if (lane < kIcpTerms) partial[warp * kIcpTerms + lane] = acc;
}

// Fixed-order sum of the per-warp partials: thread l adds column l top to bottom.
__global__ void icp_reduce_kernel(const double* __restrict__ partial, int64_t warps, double* __restrict__ sums) {
  const int l = threadIdx.x;
  if (l >= kIcpTerms) return;
  double s = 0.0;
  for (int64_t w = 0; w < warps; ++w) s += partial[w * kIcpTerms + l];
  sums[l] = s;
}

}  // namespace sf

using namespace sf;

extern "C" int sf_ransac_count_inliers(const double* a, const double* b, int64_t m, const double* transforms,
                                       int64_t n_draws, double threshold, int32_t* counts, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(m >= 0 && n_draws >= 0 && n_draws < (int64_t(1) << 31), SF_ERR_ARG, "sf_ransac_count_inliers: bad sizes");
  if (n_draws == 0) return SF_OK;
  SF_REQUIRE(transforms && counts && (m == 0 || (a && b)), SF_ERR_ARG, "sf_ransac_count_inliers: null argument");
  ransac_inliers_kernel<<<unsigned(n_draws), 256, 0, stream>>>(a, b, m, transforms, threshold, counts);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_icp_plane_step(sf_grid* g, const double* scan, int64_t n_scan, const double* transform_host,
                                 double d_max, double* sums_host, int32_t* nearest, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0 && g->has_normals, SF_ERR_ARG, "sf_icp_plane_step: grid built without normals");
  SF_REQUIRE(scan && transform_host && sums_host && n_scan >= 0, SF_ERR_ARG, "sf_icp_plane_step: null argument");
  SF_REQUIRE(radius_fits(g, d_max), SF_ERR_ARG,
             "sf_icp_plane_step: d_max %g exceeds the cell edge %g the grid was built for", d_max, g->cell);
  for (int k = 0; k < kIcpTerms; ++k) sums_host[k] = 0.0;
  if (n_scan == 0) return SF_OK;
  const int64_t blocks = std::min<int64_t>((n_scan * 32 + 255) / 256, 148 * 8);
  const int64_t warps = blocks * 8;
  double *transform = nullptr, *partial = nullptr, *sums = nullptr;
  Scratch scratch(stream);
  SF_CUDA(scratch.alloc(&transform, 12 * sizeof(double)));
  SF_CUDA(scratch.alloc(&partial, size_t(warps) * kIcpTerms * sizeof(double)));
  SF_CUDA(scratch.alloc(&sums, kIcpTerms * sizeof(double)));
  SF_CUDA(cudaMemcpyAsync(transform, transform_host, 12 * sizeof(double), cudaMemcpyHostToDevice, stream));
  icp_plane_kernel<<<unsigned(blocks), 256, 0, stream>>>(g->view(), scan, n_scan, transform, d_max, partial, nearest);
  icp_reduce_kernel<<<1, 32, 0, stream>>>(partial, warps, sums);
  SF_CUDA(cudaGetLastError());
  SF_CUDA(cudaMemcpyAsync(sums_host, sums, kIcpTerms * sizeof(double), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  return SF_OK;
}
