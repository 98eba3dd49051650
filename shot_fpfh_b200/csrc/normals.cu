// "Next" row #2 of SURVEY.md §8f: PCA normals, `compute_normals` (descriptors/pca_based_descriptors.py:15-59), which
// `get_data` runs on every cloud before the hot path (io_ply.py:259-301, k = 30). It reuses the hot path's grid and
// its LAPACK-path 3x3 eigensolver (the normal is np.linalg.eigh(cov)[1][:, 0]: without `pre_computed_normals` its
// sign is LAPACK's, which sf_eigh3.cuh reproduces).
//   knn_kernel         <- KDTree(cloud).query(queries, k, return_distance=False)  (pca_based_descriptors.py:46)
//   pca_normal_kernel  <- pca(cloud[neighbourhood])[1][:, 0] + reorientation      (pca_based_descriptors.py:15-26, :51-57)
#include "sf_common.cuh"

namespace sf {

constexpr int kKnnCapacity = 512;  // candidates within one cell edge of the query that a warp can rank

// One warp per query. All cloud points within `reach` (<= cell edge, so they all lie in the 27 surrounding cells) are
// collected with their float64 squared distances; if there are at least k of them the k nearest are among them and
// are extracted by k rounds of warp-wide arg-min (ties: lower cell-sorted position). Otherwise the query is flagged
// and the host retries it with a larger reach.
__global__ void __launch_bounds__(128)
    knn_kernel(GridView g, const double* __restrict__ queries, int64_t nq, int k, double reach2,
               int32_t* __restrict__ nbr_index, int32_t* __restrict__ status) {
  __shared__ double cand_d[4][kKnnCapacity];
  __shared__ int32_t cand_i[4][kKnnCapacity];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t q = blockIdx.x * int64_t(4) + warp;
  if (q >= nq) return;
  if (status[q] == 1) return;  // already solved by a previous (smaller-reach) attempt
  const double qx = __ldg(queries + 3 * q), qy = __ldg(queries + 3 * q + 1), qz = __ldg(queries + 3 * q + 2);
  const Runs runs = build_runs(g, qx, qy, qz, lane);
  const int total = runs.pref[9];
  int count = 0;
  bool overflow = false;
  for (int base = 0; base < total; base += 32) {
    const int v = base + lane;
    bool hit = false;
    int pos = 0;
    double d2 = 0.0;
    if (v < total) {
      pos = run_position(runs, v);
      const double4 p = load_pt(g.pts + pos);
      d2 = rdist3(qx - p.x, qy - p.y, qz - p.z);
      hit = d2 <= reach2;
    }
    const unsigned mask = __ballot_sync(kFull, hit);
    const int slot = count + __popc(mask & lanemask_lt());
    if (hit) {
      if (slot < kKnnCapacity) { cand_d[warp][slot] = d2; cand_i[warp][slot] = pos; }
      else overflow = true;
    }
    count += __popc(mask);
  }
  overflow = __any_sync(kFull, overflow);
  __syncwarp();
  if (count < k || overflow) {  // not enough points within reach (or too many to rank): retry with another reach
    if (lane == 0) status[q] = overflow ? 2 : 0;
    return;
  }
  for (int r = 0; r < k; ++r) {
    double best = INFINITY;
    int best_slot = -1, best_pos = 0x7fffffff;
    for (int s = lane; s < count; s += 32) {
      const double d = cand_d[warp][s];
      const int p = cand_i[warp][s];
      if (d < best || (d == best && p < best_pos)) { best = d; best_slot = s; best_pos = p; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(kFull, best, o);
      const int os = __shfl_xor_sync(kFull, best_slot, o);
      const int op = __shfl_xor_sync(kFull, best_pos, o);
      if (od < best || (od == best && op < best_pos)) { best = od; best_slot = os; best_pos = op; }
    }
    if (lane == 0) {  // original point index (the grid may be rebuilt between attempts; positions would go stale)
      nbr_index[q * k + r] = int32_t(__double_as_longlong(load_pt(g.pts + best_pos).w));
      cand_d[warp][best_slot] = INFINITY;
    }
    __syncwarp();
  }
  if (lane == 0) status[q] = 1;
}

// One warp per batch of 32 queries (same structure as shot_lrf_kernel): covariance of the neighbourhood about its
// barycentre by warp reduction, one eigen-decomposition per lane, eigenvector of the smallest eigenvalue.
__global__ void __launch_bounds__(128)
    pca_normal_kernel(const double* __restrict__ xyz, int64_t nq, const int64_t* __restrict__ offsets, int fixed_k,
                      const int32_t* __restrict__ nbr, const double* __restrict__ pre_normals,
                      double* __restrict__ normals) {
  const int lane = threadIdx.x & 31;
  const int64_t q0 = ((blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5) * 32;
  if (q0 >= nq) return;
  const int batch = int(nq - q0 < 32 ? nq - q0 : 32);
  const int64_t mine = q0 + (lane < batch ? lane : 0);
  const int64_t my_begin = offsets ? __ldg(offsets + mine) : mine * fixed_k;
  const int64_t my_end = offsets ? __ldg(offsets + mine + 1) : (mine + 1) * fixed_k;
  double cov[6] = {0, 0, 0, 0, 0, 0};
  for (int j = 0; j < batch; ++j) {
    const int64_t begin = __shfl_sync(kFull, my_begin, j), end = __shfl_sync(kFull, my_end, j);
    const double n = double(end - begin);
    double sx = 0, sy = 0, sz = 0;
    for (int64_t i = begin + lane; i < end; i += 32) {
      const double* p = xyz + 3 * int64_t(__ldg(nbr + i));
      sx += __ldg(p); sy += __ldg(p + 1); sz += __ldg(p + 2);
    }
    const double mx = warp_sum(sx) / n, my = warp_sum(sy) / n, mz = warp_sum(sz) / n;
    double m[6] = {0, 0, 0, 0, 0, 0};
    for (int64_t i = begin + lane; i < end; i += 32) {
      const double* p = xyz + 3 * int64_t(__ldg(nbr + i));
      const double cx = __ldg(p) - mx, cy = __ldg(p + 1) - my, cz = __ldg(p + 2) - mz;
      m[0] += cx * cx; m[1] += cx * cy; m[2] += cx * cz;
      m[3] += cy * cy; m[4] += cy * cz; m[5] += cz * cz;
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const double v = warp_sum(m[c]) / n;
      if (lane == j) cov[c] = v;
    }
  }
  if (lane < batch) {
    double nx = 0, ny = 0, nz = 0;  // an empty neighbourhood (radius variant) would make NumPy produce NaNs
    if (my_end > my_begin) {
      double eval[3], evec[3][3];
      eigh3(cov, eval, evec);
      nx = evec[0][0]; ny = evec[0][1]; nz = evec[0][2];
      if (pre_normals != nullptr) {
        const double dot = nx * pre_normals[3 * mine] + ny * pre_normals[3 * mine + 1] + nz * pre_normals[3 * mine + 2];
        if (dot < 0.0) { nx = -nx; ny = -ny; nz = -nz; }
      }
    } else {
      nx = ny = nz = __longlong_as_double(0x7ff8000000000000ll);
    }
    normals[3 * mine] = nx;
    normals[3 * mine + 1] = ny;
    normals[3 * mine + 2] = nz;
  }
}

}  // namespace sf

using namespace sf;

extern "C" int sf_knn(sf_grid* g, const double* queries, int64_t nq, int32_t k, double reach, int32_t* nbr_index,
                      int32_t* status, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_knn: grid not built");
  SF_REQUIRE(queries && nbr_index && status && nq >= 0, SF_ERR_ARG, "sf_knn: bad arguments");
  SF_REQUIRE(k >= 1 && k <= kKnnCapacity, SF_ERR_CAPACITY, "sf_knn: k must be in [1, %d]", kKnnCapacity);
  SF_REQUIRE(radius_fits(g, reach), SF_ERR_ARG, "sf_knn: reach exceeds the grid's cell edge");
  if (nq == 0) return SF_OK;
  knn_kernel<<<unsigned((nq + 3) / 4), 128, 0, stream>>>(g->view(), queries, nq, k, reach * reach, nbr_index, status);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_pca_normals(const double* xyz, int64_t nq, const int64_t* offsets, int32_t fixed_k,
                              const int32_t* nbr_index, const double* pre_normals, double* normals, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(xyz && nbr_index && normals && nq >= 0 && (offsets != nullptr || fixed_k >= 1), SF_ERR_ARG,
             "sf_pca_normals: bad arguments");
  if (nq == 0) return SF_OK;
  const int64_t warps = (nq + 31) / 32;
  pca_normal_kernel<<<unsigned((warps + 3) / 4), 128, 0, stream>>>(xyz, nq, offsets, fixed_k, nbr_index, pre_normals,
                                                                  normals);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}
