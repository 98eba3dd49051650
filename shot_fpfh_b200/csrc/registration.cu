// Registration stages downstream of the matcher (SURVEY.md §8f row 4), the data-parallel part of each:
//   RANSAC  (matching/ransac.py:17-82)  the n_draws x n_matches inlier count — the draws replay NumPy's generator on
//           the host and the 4-point Kabsch fits are a batched host SVD; what costs is the count (:55-62).
//   ICP     (icp.py:137-189, core/solvers.py:34-48)  per iteration: transform the subsampled scan, nearest reference
//           point within d_max of each (KDTree.query + the `<= d_max` filter), and the sums of the point-to-plane
//           normal equations g^T g, g^T h plus the residual — one kernel, one 29-double result per iteration.
//   Adaptive RANSAC (matching/ransac.py ransac_on_matches_adaptive; no counterpart in the reference) draws, checks, fits
//           and scores its 3-match hypotheses here in batches of 2^20; only the refit on the inliers is on the host.
#include <algorithm>

#include "sf_common.cuh"

namespace sf {

// ---- RANSAC: inliers of every candidate transform ------------------------------------------------------------
// The inlier predicate of every RANSAC kernel: match (a, b) is an inlier of {R row-major (9), t (3)} when
// sqrt(ransac_residual_sq(...)) <= threshold (ransac.py:55-62; np.linalg.norm, i.e. the sqrt is taken before
// comparing). IEEE sqrt is correctly rounded and monotone, so `residual_sq <= T` with T the largest double whose sqrt
// is <= threshold (inlier_threshold_sq) is the same predicate without the sqrt.
__device__ __forceinline__ double ransac_residual_sq(const double r[9], const double t[3], double ax, double ay,
                                                     double az, double bx, double by, double bz) {
  const double dx = (r[0] * ax + r[1] * ay + r[2] * az + t[0]) - bx;
  const double dy = (r[3] * ax + r[4] * ay + r[5] * az + t[1]) - by;
  const double dz = (r[6] * ax + r[7] * ay + r[8] * az + t[2]) - bz;
  return dx * dx + dy * dy + dz * dz;
}

// One block per draw. transforms[d] = {R row-major (9), t (3)}.
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
    count += sqrt(ransac_residual_sq(r, t, __ldg(a + 3 * i), __ldg(a + 3 * i + 1), __ldg(a + 3 * i + 2),
                                     __ldg(b + 3 * i), __ldg(b + 3 * i + 1), __ldg(b + 3 * i + 2))) <= threshold;
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

// ---- Adaptive RANSAC: device-drawn 3-point hypotheses (oracle/adaptive_ransac_oracle.py is the specification) -----
// Per batch of kAdaptiveBatch draws: draw + edge check (thread per draw, survivors compacted), Kabsch + self-check
// (thread per survivor, valid hypotheses compacted), scoring (hypotheses x matches), then the 64-bit winner key
// (count << 32) | (0xFFFFFFFF - draw), which carries across batches and sends ties to the lowest draw.
constexpr int64_t kAdaptiveBatch = int64_t(1) << 20;
constexpr uint64_t kGoldenGamma = 0x9E3779B97F4A7C15ull;
constexpr double kDegenerate = 1e-12;

__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// The three distinct match indices of draw d (base = seed * kGoldenGamma, m < 2^32 so every product fits 64 bits).
__device__ __forceinline__ void draw_triple(uint64_t base, uint64_t d, uint64_t m, uint32_t j[3]) {
  const uint64_t x = base + 3 * d;
  const uint64_t j0 = ((splitmix64(x) >> 32) * m) >> 32;
  uint64_t j1 = ((splitmix64(x + 1) >> 32) * (m - 1)) >> 32;
  j1 += j1 >= j0;
  uint64_t j2 = ((splitmix64(x + 2) >> 32) * (m - 2)) >> 32;
  j2 += j2 >= (j0 < j1 ? j0 : j1);
  j2 += j2 >= (j0 < j1 ? j1 : j0);
  j[0] = uint32_t(j0); j[1] = uint32_t(j1); j[2] = uint32_t(j2);
}

__device__ __forceinline__ void load_triple(const double* __restrict__ p, const uint32_t j[3], double out[3][3]) {
#pragma unroll
  for (int s = 0; s < 3; ++s)
#pragma unroll
    for (int c = 0; c < 3; ++c) out[s][c] = __ldg(p + 3 * int64_t(j[s]) + c);
}

__device__ __forceinline__ double length3(const double p[3], const double q[3]) {
  return sqrt(rdist3(p[0] - q[0], p[1] - q[1], p[2] - q[2]));
}

// min(|a_p - a_q|, |b_p - b_q|) >= edge_similarity * max(...) for the three pairs.
__device__ __forceinline__ bool edges_consistent(const double pa[3][3], const double pb[3][3], double edge_similarity) {
  bool ok = true;
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    const int p = e == 2 ? 1 : 0, q = e == 0 ? 1 : 2;
    const double la = length3(pa[p], pa[q]), lb = length3(pb[p], pb[q]);
    ok &= fmin(la, lb) >= edge_similarity * fmax(la, lb);
  }
  return ok;
}

// ((x0 y0 + x1 y1) + x2 y2), every operation rounded on its own.
__device__ __forceinline__ double dot3_rn(double x0, double x1, double x2, double y0, double y1, double y2) {
  return add_rn(add_rn(mul_rn(x0, y0), mul_rn(x1, y1)), mul_rn(x2, y2));
}

__device__ __forceinline__ void cross_rn(const double x[3], const double y[3], double out[3]) {
  out[0] = add_rn(mul_rn(x[1], y[2]), -mul_rn(x[2], y[1]));
  out[1] = add_rn(mul_rn(x[2], y[0]), -mul_rn(x[0], y[2]));
  out[2] = add_rn(mul_rn(x[0], y[1]), -mul_rn(x[1], y[0]));
}

// Kabsch on three pairs through eigh3(H^T H) (the oracle's step 3, operation for operation); false when degenerate.
__device__ bool kabsch3(const double pa[3][3], const double pb[3][3], double tr[12]) {
  double abar[3], bbar[3], ac[3][3], bc[3][3], h[3][3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    abar[c] = add_rn(add_rn(pa[0][c], pa[1][c]), pa[2][c]) / 3.0;
    bbar[c] = add_rn(add_rn(pb[0][c], pb[1][c]), pb[2][c]) / 3.0;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      ac[s][c] = add_rn(pa[s][c], -abar[c]);
      bc[s][c] = add_rn(pb[s][c], -bbar[c]);
    }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) h[i][j] = dot3_rn(ac[0][i], ac[1][i], ac[2][i], bc[0][j], bc[1][j], bc[2][j]);
  // M = H^T H, lower triangle {m00, m10, m20, m11, m21, m22}
  auto col_dot = [&](int i, int j) { return dot3_rn(h[0][i], h[1][i], h[2][i], h[0][j], h[1][j], h[2][j]); };
  const double mtm[6] = {col_dot(0, 0), col_dot(1, 0), col_dot(2, 0), col_dot(1, 1), col_dot(2, 1), col_dot(2, 2)};
  double lam[3], vec[3][3];
  eigh3(mtm, lam, vec);
  if (lam[1] <= kDegenerate * lam[2]) return false;
  double u[3][3], v[3][3];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const double* vk = vec[2 - k];
    double hv[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      v[k][i] = vk[i];
      hv[i] = dot3_rn(h[i][0], h[i][1], h[i][2], vk[0], vk[1], vk[2]);
    }
    const double norm = sqrt(dot3_rn(hv[0], hv[1], hv[2], hv[0], hv[1], hv[2]));
#pragma unroll
    for (int i = 0; i < 3; ++i) u[k][i] = hv[i] / norm;
  }
  cross_rn(u[0], u[1], u[2]);
  cross_rn(v[0], v[1], v[2]);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) tr[3 * i + j] = dot3_rn(v[0][i], v[1][i], v[2][i], u[0][j], u[1][j], u[2][j]);
#pragma unroll
  for (int i = 0; i < 3; ++i)
    tr[9 + i] = add_rn(bbar[i], -dot3_rn(tr[3 * i], tr[3 * i + 1], tr[3 * i + 2], abar[0], abar[1], abar[2]));
  return true;
}

// Warp-aggregated append: the lanes with `keep` get consecutive slots of a list whose length is *counter.
__device__ __forceinline__ uint32_t warp_append(bool keep, uint32_t* counter) {
  const unsigned mask = __ballot_sync(kFull, keep);
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(mask) - 1;
  uint32_t first = 0;
  if (mask != 0 && lane == leader) first = atomicAdd(counter, uint32_t(__popc(mask)));
  first = __shfl_sync(kFull, first, leader < 0 ? 0 : leader);
  return first + uint32_t(__popc(mask & ((1u << lane) - 1u)));
}

// counters[0] = survivors of the edge check, counters[1] = valid hypotheses.
__global__ void __launch_bounds__(256)
    ransac_draw_kernel(const double* __restrict__ a, const double* __restrict__ b, uint64_t m, uint64_t base,
                       uint64_t first, uint32_t n, double edge_similarity, uint32_t* __restrict__ survivors,
                       uint32_t* __restrict__ counters) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  bool pass = false;
  if (i < n) {
    uint32_t j[3];
    draw_triple(base, first + i, m, j);
    double pa[3][3], pb[3][3];
    load_triple(a, j, pa);
    load_triple(b, j, pb);
    pass = edges_consistent(pa, pb, edge_similarity);
  }
  const uint32_t slot = warp_append(pass, &counters[0]);
  if (pass) survivors[slot] = uint32_t(first + i);
}

// One thread per survivor (the grid covers the whole batch; threads past counters[0] only take part in the append).
__global__ void __launch_bounds__(128)
    ransac_fit_kernel(const double* __restrict__ a, const double* __restrict__ b, uint64_t m, uint64_t base,
                      const uint32_t* __restrict__ survivors, double t_sq, uint32_t* __restrict__ counters,
                      uint32_t* __restrict__ valid_draws, double* __restrict__ transforms) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x * blockDim.x >= counters[0]) return;  // uniform per block: whole warps leave together
  bool valid = false;
  uint32_t d = 0;
  double tr[12];
  if (i < counters[0]) {
    d = survivors[i];
    uint32_t j[3];
    draw_triple(base, d, m, j);
    double pa[3][3], pb[3][3];
    load_triple(a, j, pa);
    load_triple(b, j, pb);
    valid = kabsch3(pa, pb, tr);
#pragma unroll
    for (int s = 0; s < 3; ++s)  // Open3D's distance checker: the draw's own pairs are inliers of its transform
      valid = valid && ransac_residual_sq(tr, tr + 9, pa[s][0], pa[s][1], pa[s][2], pb[s][0], pb[s][1], pb[s][2]) <= t_sq;
  }
  const uint32_t slot = warp_append(valid, &counters[1]);
  if (valid) {
    valid_draws[slot] = d;
#pragma unroll
    for (int k = 0; k < 12; ++k) transforms[12 * int64_t(slot) + k] = tr[k];
  }
}

// Thread = hypothesis (transform in registers), blockIdx.y = a chunk of the matches, staged through shared memory in
// tiles that every thread reads as broadcasts. Partial counts meet in an integer atomicAdd: exact, order-free.
constexpr int kScoreThreads = 256;
__global__ void __launch_bounds__(kScoreThreads)
    ransac_score_kernel(const double* __restrict__ a, const double* __restrict__ b, int64_t m, int64_t chunk,
                        const double* __restrict__ transforms, uint32_t n_valid, double t_sq,
                        int32_t* __restrict__ counts) {
  __shared__ double sa[3 * kScoreThreads], sb[3 * kScoreThreads];
  const uint32_t h = blockIdx.x * kScoreThreads + threadIdx.x;
  const bool live = h < n_valid;
  double r[9], t[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) r[k] = live ? transforms[12 * int64_t(h) + k] : 0.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) t[k] = live ? transforms[12 * int64_t(h) + 9 + k] : 0.0;
  const int64_t begin = int64_t(blockIdx.y) * chunk, end = std::min<int64_t>(m, begin + chunk);
  int count = 0;
  for (int64_t s = begin; s < end; s += kScoreThreads) {
    const int n = int(std::min<int64_t>(kScoreThreads, end - s));
    __syncthreads();
    for (int k = threadIdx.x; k < 3 * n; k += kScoreThreads) {
      sa[k] = __ldg(a + 3 * s + k);
      sb[k] = __ldg(b + 3 * s + k);
    }
    __syncthreads();
    if (live)
      for (int k = 0; k < n; ++k)
        count += ransac_residual_sq(r, t, sa[3 * k], sa[3 * k + 1], sa[3 * k + 2], sb[3 * k], sb[3 * k + 1],
                                    sb[3 * k + 2]) <= t_sq;
  }
  if (live && count) atomicAdd(&counts[h], count);
}

__device__ __forceinline__ unsigned long long winner_key(int32_t count, uint32_t draw) {
  return (static_cast<unsigned long long>(count) << 32) | (0xFFFFFFFFull - draw);
}

__global__ void __launch_bounds__(256)
    ransac_best_kernel(const uint32_t* __restrict__ valid_draws, const int32_t* __restrict__ counts, uint32_t n_valid,
                       unsigned long long* __restrict__ best) {
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long key = h < n_valid ? winner_key(counts[h], valid_draws[h]) : 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(kFull, key, o);
    key = other > key ? other : key;
  }
  if ((threadIdx.x & 31) == 0 && key != 0) atomicMax(best, key);
}

// After ransac_best_kernel: the hypothesis of this batch that holds the winner key (if any) copies its transform.
__global__ void __launch_bounds__(256)
    ransac_keep_kernel(const uint32_t* __restrict__ valid_draws, const int32_t* __restrict__ counts, uint32_t n_valid,
                       const double* __restrict__ transforms, const unsigned long long* __restrict__ best,
                       double* __restrict__ best_transform) {
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h < n_valid && winner_key(counts[h], valid_draws[h]) == *best)
    for (int k = 0; k < 12; ++k) best_transform[k] = transforms[12 * int64_t(h) + k];
}

__global__ void __launch_bounds__(256)
    ransac_mask_kernel(const double* __restrict__ a, const double* __restrict__ b, int64_t m,
                       const double* __restrict__ transform, double t_sq, uint8_t* __restrict__ mask) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= m) return;
  double r[9], t[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) r[k] = __ldg(transform + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) t[k] = __ldg(transform + 9 + k);
  mask[i] = ransac_residual_sq(r, t, __ldg(a + 3 * i), __ldg(a + 3 * i + 1), __ldg(a + 3 * i + 2), __ldg(b + 3 * i),
                               __ldg(b + 3 * i + 1), __ldg(b + 3 * i + 2)) <= t_sq;
}

// The largest double whose sqrt is <= threshold.
double inlier_threshold_sq(double threshold) {
  double t = threshold * threshold;
  while (std::sqrt(t) > threshold) t = std::nextafter(t, 0.0);
  while (std::sqrt(std::nextafter(t, INFINITY)) <= threshold) t = std::nextafter(t, INFINITY);
  return t;
}

// Device buffers of one batch, sized for kAdaptiveBatch draws.
struct AdaptiveBatch {
  uint32_t* survivors;
  uint32_t* valid_draws;
  double* transforms;
  int32_t* counts;
  uint32_t* counters;  // [2]
};

// Draws [first, first + n): survivors, valid hypotheses with their transforms, and their inlier counts.
// One host synchronisation (the counters); n_host = {survivors, valid}.
int adaptive_batch(const double* a, const double* b, int64_t m, double t_sq, double edge_similarity, uint64_t base,
                   int64_t first, int64_t n, const AdaptiveBatch& buf, int64_t n_host[2], cudaStream_t stream) {
  SF_CUDA(cudaMemsetAsync(buf.counters, 0, 2 * sizeof(uint32_t), stream));
  const unsigned draw_blocks = unsigned((n + 255) / 256);
  ransac_draw_kernel<<<draw_blocks, 256, 0, stream>>>(a, b, uint64_t(m), base, uint64_t(first), uint32_t(n),
                                                       edge_similarity, buf.survivors, buf.counters);
  ransac_fit_kernel<<<unsigned((n + 127) / 128), 128, 0, stream>>>(a, b, uint64_t(m), base, buf.survivors, t_sq,
                                                                    buf.counters, buf.valid_draws, buf.transforms);
  SF_CUDA(cudaGetLastError());
  uint32_t counters[2];
  SF_CUDA(cudaMemcpyAsync(counters, buf.counters, sizeof(counters), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  n_host[0] = counters[0];
  n_host[1] = counters[1];
  const uint32_t n_valid = counters[1];
  if (n_valid == 0) return SF_OK;
  SF_CUDA(cudaMemsetAsync(buf.counts, 0, n_valid * sizeof(int32_t), stream));
  // enough blocks to fill the GPU: the matches are split into chunks (multiples of the staging tile) along y
  const int64_t hyp_blocks = (n_valid + kScoreThreads - 1) / kScoreThreads;
  const int64_t tiles = (m + kScoreThreads - 1) / kScoreThreads;
  const int64_t splits = std::max<int64_t>(1, std::min<int64_t>(tiles, (148 * 8 + hyp_blocks - 1) / hyp_blocks));
  const int64_t chunk = (tiles + splits - 1) / splits * kScoreThreads;
  const dim3 grid(unsigned(hyp_blocks), unsigned((m + chunk - 1) / chunk));
  ransac_score_kernel<<<grid, kScoreThreads, 0, stream>>>(a, b, m, chunk, buf.transforms, n_valid, t_sq, buf.counts);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

// Checks shared by both entry points.
int adaptive_arguments(const char* fn, const double* a, const double* b, int64_t m, double threshold,
                       double edge_similarity) {
  SF_REQUIRE(a && b, SF_ERR_ARG, "%s: null argument", fn);
  SF_REQUIRE(m >= 3 && m <= int64_t(0xFFFFFFFF), SF_ERR_ARG, "%s: %lld matches (3 .. 2^32 - 1)", fn, (long long)m);
  SF_REQUIRE(threshold > 0.0 && std::isfinite(threshold), SF_ERR_ARG, "%s: threshold %g", fn, threshold);
  SF_REQUIRE(edge_similarity > 0.0 && edge_similarity <= 1.0, SF_ERR_ARG, "%s: edge_similarity %g outside (0, 1]", fn,
             edge_similarity);
  return SF_OK;
}

int adaptive_alloc(Scratch& scratch, int64_t capacity, AdaptiveBatch& buf) {
  SF_CUDA(scratch.alloc(&buf.survivors, size_t(capacity) * sizeof(uint32_t)));
  SF_CUDA(scratch.alloc(&buf.valid_draws, size_t(capacity) * sizeof(uint32_t)));
  SF_CUDA(scratch.alloc(&buf.transforms, size_t(capacity) * 12 * sizeof(double)));
  SF_CUDA(scratch.alloc(&buf.counts, size_t(capacity) * sizeof(int32_t)));
  SF_CUDA(scratch.alloc(&buf.counters, 2 * sizeof(uint32_t)));
  return SF_OK;
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

extern "C" int sf_ransac_adaptive(const double* a, const double* b, int64_t m, double threshold, double edge_similarity,
                                  uint64_t seed, int64_t max_draws, double confidence, double* transform_host,
                                  int64_t* best_draw_host, int64_t* best_count_host, int64_t* draws_used_host,
                                  int64_t* valid_host, uint8_t* inlier_mask, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int status = adaptive_arguments("sf_ransac_adaptive", a, b, m, threshold, edge_similarity);
  if (status != SF_OK) return status;
  SF_REQUIRE(transform_host && best_draw_host && best_count_host && draws_used_host && valid_host && inlier_mask,
             SF_ERR_ARG, "sf_ransac_adaptive: null argument");
  SF_REQUIRE(max_draws >= 1 && max_draws <= int64_t(0xFFFFFFFF), SF_ERR_ARG,
             "sf_ransac_adaptive: max_draws %lld outside [1, 2^32 - 1]", (long long)max_draws);
  SF_REQUIRE(confidence > 0.0 && confidence < 1.0, SF_ERR_ARG, "sf_ransac_adaptive: confidence %g outside (0, 1)",
             confidence);
  const double t_sq = inlier_threshold_sq(threshold);
  const uint64_t base = seed * kGoldenGamma;
  const double log_miss = std::log(1.0 - confidence);
  Scratch scratch(stream);
  AdaptiveBatch buf;
  int s = adaptive_alloc(scratch, std::min<int64_t>(kAdaptiveBatch, max_draws), buf);
  if (s != SF_OK) return s;
  unsigned long long* best = nullptr;  // the winner key, then the winner's transform (12 doubles)
  SF_CUDA(scratch.alloc(&best, 13 * sizeof(double)));
  double* best_transform = reinterpret_cast<double*>(best + 1);
  SF_CUDA(cudaMemsetAsync(best, 0, sizeof(unsigned long long), stream));
  unsigned long long key = 0;
  int64_t k = 0, valid = 0;
  while (true) {
    const int64_t first = k * kAdaptiveBatch, n = std::min<int64_t>(kAdaptiveBatch, max_draws - first);
    int64_t counters[2];
    s = adaptive_batch(a, b, m, t_sq, edge_similarity, base, first, n, buf, counters, stream);
    if (s != SF_OK) return s;
    valid += counters[1];
    if (counters[1] > 0) {
      const unsigned blocks = unsigned((counters[1] + 255) / 256);
      ransac_best_kernel<<<blocks, 256, 0, stream>>>(buf.valid_draws, buf.counts, uint32_t(counters[1]), best);
      ransac_keep_kernel<<<blocks, 256, 0, stream>>>(buf.valid_draws, buf.counts, uint32_t(counters[1]),
                                                      buf.transforms, best, best_transform);
      SF_CUDA(cudaGetLastError());
      SF_CUDA(cudaMemcpyAsync(&key, best, sizeof(key), cudaMemcpyDeviceToHost, stream));
      SF_CUDA(cudaStreamSynchronize(stream));
    }
    ++k;
    if (k * kAdaptiveBatch >= max_draws) break;
    const double c = double(key >> 32);  // stop once k B draws miss an all-inlier triple with probability <= 1 - confidence
    const double r = c / double(m);
    if (c > 0 && double(k * kAdaptiveBatch) * std::log1p(-(r * r * r)) <= log_miss) break;
  }
  *draws_used_host = std::min<int64_t>(k * kAdaptiveBatch, max_draws);
  *valid_host = valid;
  *best_count_host = int64_t(key >> 32);
  *best_draw_host = key ? int64_t(0xFFFFFFFFull - (key & 0xFFFFFFFFull)) : -1;
  if (key == 0) {
    for (int i = 0; i < 12; ++i) transform_host[i] = 0.0;
    SF_CUDA(cudaMemsetAsync(inlier_mask, 0, size_t(m), stream));
  } else {
    ransac_mask_kernel<<<unsigned((m + 255) / 256), 256, 0, stream>>>(a, b, m, best_transform, t_sq, inlier_mask);
    SF_CUDA(cudaGetLastError());
    SF_CUDA(cudaMemcpyAsync(transform_host, best_transform, 12 * sizeof(double), cudaMemcpyDeviceToHost, stream));
  }
  SF_CUDA(cudaStreamSynchronize(stream));
  return SF_OK;
}

extern "C" int sf_ransac_adaptive_batch(const double* a, const double* b, int64_t m, double threshold,
                                        double edge_similarity, uint64_t seed, int64_t first_draw, int64_t n_draws,
                                        uint32_t* survivors, uint32_t* valid_draws, double* transforms, int32_t* counts,
                                        int64_t* n_host, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int status = adaptive_arguments("sf_ransac_adaptive_batch", a, b, m, threshold, edge_similarity);
  if (status != SF_OK) return status;
  SF_REQUIRE(survivors && valid_draws && transforms && counts && n_host, SF_ERR_ARG,
             "sf_ransac_adaptive_batch: null argument");
  SF_REQUIRE(n_draws >= 1 && n_draws <= kAdaptiveBatch && first_draw >= 0 &&
                 first_draw + n_draws <= int64_t(0xFFFFFFFF),
             SF_ERR_ARG, "sf_ransac_adaptive_batch: draws [%lld, +%lld) outside [0, 2^32 - 1) or over one batch",
             (long long)first_draw, (long long)n_draws);
  Scratch scratch(stream);
  AdaptiveBatch buf{survivors, valid_draws, transforms, counts, nullptr};
  SF_CUDA(scratch.alloc(&buf.counters, 2 * sizeof(uint32_t)));
  const int s = adaptive_batch(a, b, m, inlier_threshold_sq(threshold), edge_similarity, seed * kGoldenGamma,
                               first_draw, n_draws, buf, n_host, stream);
  if (s != SF_OK) return s;
  SF_CUDA(cudaStreamSynchronize(stream));
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
