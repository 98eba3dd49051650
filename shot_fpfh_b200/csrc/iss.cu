// Kernel group K: ISS salient keypoints (Intrinsic Shape Signatures, Zhong 2009). The reference has no keypoint
// detector of this kind; the specification is the restatement in oracle/iss_oracle.py (Open3D's definition, covariance
// accumulated about the point). Both passes run on ONE grid built for max(salient radius, non-max radius): the culled
// runs (build_runs with r2) drop the cells out of reach of the smaller radius, and the saliency stays in cell-sorted
// order, so the non-maximum pass reads s_j by position with no permutation.
//   iss_saliency_kernel  every point: n_i, the covariance of N_s(i) about p_i, eigh3 (the dsyevd path), the ratio tests
//   iss_nms_kernel       every point with s > 0: |N_n(i)| >= m and no s_j > s_i in N_n(i), flag at the original index
// then DeviceSelect::Flagged over a counting iterator lists the flagged original indices in ascending order (no sort).
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <cmath>

#include "sf_common.cuh"
#include "sf_eigh3.cuh"

namespace sf {

// One warp per 32 consecutive cell-sorted points (the batching of pca_normal_kernel): for each of them in turn, all 32
// lanes scan its candidates (the walk of knn_kernel) and accumulate n_i and the 3 + 6 sums of the offsets c = p_j - p_i;
// the warp sums land in the lane that owns the point, and then every lane solves its own 3x3 problem.
__global__ void __launch_bounds__(128)
    iss_saliency_kernel(GridView g, double r2, int min_neighbors, double gamma_21, double gamma_32,
                        double* __restrict__ saliency, int32_t* __restrict__ counts, double* __restrict__ eigvals) {
  const int lane = threadIdx.x & 31;
  const int64_t p0 = ((blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5) * 32;
  if (p0 >= g.n) return;
  const int batch = int(g.n - p0 < 32 ? g.n - p0 : 32);
  const int64_t mine = p0 + (lane < batch ? lane : 0);
  const double4 me = load_pt(g.pts + mine);
  int my_count = 0;
  double my_sum[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // x y z, xx xy xz yy yz zz
  for (int j = 0; j < batch; ++j) {
    const double qx = __shfl_sync(kFull, me.x, j), qy = __shfl_sync(kFull, me.y, j), qz = __shfl_sync(kFull, me.z, j);
    const Runs runs = build_runs(g, qx, qy, qz, lane, r2);
    const int total = runs.pref[9];
    int count = 0;
    double s[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int v = lane; v < total; v += 32) {
      const double4 p = load_pt(g.pts + run_position(runs, v));
      const double dx = p.x - qx, dy = p.y - qy, dz = p.z - qz;
      if (rdist3(dx, dy, dz) <= r2) {
        ++count;
        s[0] += dx; s[1] += dy; s[2] += dz;
        s[3] += dx * dx; s[4] += dx * dy; s[5] += dx * dz;
        s[6] += dy * dy; s[7] += dy * dz; s[8] += dz * dz;
      }
    }
    count = warp_sum(count);
    if (lane == j) my_count = count;
#pragma unroll
    for (int c = 0; c < 9; ++c) {
      const double t = warp_sum(s[c]);
      if (lane == j) my_sum[c] = t;
    }
  }
  if (lane >= batch) return;
  const double n = double(my_count);  // >= 1: the point itself
  const double mx = my_sum[0] / n, my = my_sum[1] / n, mz = my_sum[2] / n;
  // lower triangle {a11, a21, a31, a22, a32, a33}
  const double cov[6] = {my_sum[3] / n - mx * mx, my_sum[4] / n - mx * my, my_sum[5] / n - mx * mz,
                         my_sum[6] / n - my * my, my_sum[7] / n - my * mz, my_sum[8] / n - mz * mz};
  double e[3], evec[3][3];
  eigh3(cov, e, evec);  // ascending: e[0] = e3 <= e[1] = e2 <= e[2] = e1
  // IEEE float64 divisions; a NaN quotient (0 / 0: all-coincident neighbourhood) fails its comparison
  const bool salient = my_count >= min_neighbors && e[1] / e[2] < gamma_21 && e[0] / e[1] < gamma_32;
  saliency[mine] = salient ? e[0] : 0.0;
  if (counts != nullptr) counts[mine] = my_count;
  if (eigvals != nullptr) {
    eigvals[3 * mine] = e[0];
    eigvals[3 * mine + 1] = e[1];
    eigvals[3 * mine + 2] = e[2];
  }
}

struct PositiveSaliency {
  const double* s;
  __device__ __forceinline__ bool operator()(int32_t pos) const { return s[pos] > 0.0; }
};

// One warp per candidate (cell-sorted position with s > 0), grid-stride over the device-side candidate count: walk
// N_n(i), count it, and stop as soon as some lane sees s_j > s_i. Survivors flag their ORIGINAL index.
__global__ void __launch_bounds__(256)
    iss_nms_kernel(GridView g, const double* __restrict__ saliency, const int32_t* __restrict__ cand,
                   const int32_t* __restrict__ n_cand, double r2, int min_neighbors, uint8_t* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const int64_t nc = *n_cand;
  for (int64_t q = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5; q < nc; q += warps) {
    const int pos = __ldg(cand + q);
    const double4 me = load_pt(g.pts + pos);
    const double si = __ldg(saliency + pos);
    const Runs runs = build_runs(g, me.x, me.y, me.z, lane, r2);
    const int total = runs.pref[9];
    int count = 0;
    bool beaten = false;
    for (int base = 0; base < total; base += 32) {
      const int v = base + lane;
      bool hit = false, above = false;
      if (v < total) {
        const int pj = run_position(runs, v);
        const double4 p = load_pt(g.pts + pj);
        hit = rdist3(p.x - me.x, p.y - me.y, p.z - me.z) <= r2;
        above = hit && __ldg(saliency + pj) > si;
      }
      count += __popc(__ballot_sync(kFull, hit));
      if (__any_sync(kFull, above)) {
        beaten = true;
        break;
      }
    }
    if (lane == 0 && !beaten && count >= min_neighbors) flags[int32_t(__double_as_longlong(me.w))] = 1;
  }
}

}  // namespace sf

using namespace sf;

extern "C" int sf_iss_saliency(sf_grid* g, double salient_radius, int32_t min_neighbors, double gamma_21,
                               double gamma_32, double* saliency, int32_t* counts, double* eigvals, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr, SF_ERR_ARG, "sf_iss_saliency: null grid");
  SF_REQUIRE(min_neighbors >= 1, SF_ERR_ARG, "sf_iss_saliency: min_neighbors must be >= 1");
  SF_REQUIRE(std::isfinite(gamma_21) && std::isfinite(gamma_32), SF_ERR_ARG, "sf_iss_saliency: non-finite gamma");
  if (g->n == 0) return SF_OK;  // an empty cloud: nothing to write
  SF_REQUIRE(g->pts != nullptr && g->cell_start != nullptr, SF_ERR_ARG, "sf_iss_saliency: grid not built");
  SF_REQUIRE(saliency != nullptr, SF_ERR_ARG, "sf_iss_saliency: null saliency output");
  SF_REQUIRE(radius_fits(g, salient_radius), SF_ERR_ARG,
             "sf_iss_saliency: salient radius %g not in (0, cell edge %g]", salient_radius, g->cell);
  const int64_t warps = (g->n + 31) / 32;
  iss_saliency_kernel<<<unsigned((warps + 3) / 4), 128, 0, stream>>>(
      g->view(), salient_radius * salient_radius, min_neighbors, gamma_21, gamma_32, saliency, counts, eigvals);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_iss_select(sf_grid* g, const double* saliency, double non_max_radius, int32_t min_neighbors,
                             int32_t* keypoints, int64_t* count_host, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && count_host != nullptr, SF_ERR_ARG, "sf_iss_select: null grid or count");
  SF_REQUIRE(min_neighbors >= 1, SF_ERR_ARG, "sf_iss_select: min_neighbors must be >= 1");
  *count_host = 0;
  if (g->n == 0) return SF_OK;
  SF_REQUIRE(g->pts != nullptr && g->cell_start != nullptr, SF_ERR_ARG, "sf_iss_select: grid not built");
  SF_REQUIRE(saliency != nullptr && keypoints != nullptr, SF_ERR_ARG, "sf_iss_select: null saliency or output");
  SF_REQUIRE(radius_fits(g, non_max_radius), SF_ERR_ARG,
             "sf_iss_select: non-max radius %g not in (0, cell edge %g]", non_max_radius, g->cell);
  const int n = int(g->n);
  const thrust::counting_iterator<int32_t> positions(0);
  size_t if_bytes = 0, flagged_bytes = 0;
  SF_CUDA(cub::DeviceSelect::If(nullptr, if_bytes, positions, static_cast<int32_t*>(nullptr),
                                static_cast<int32_t*>(nullptr), n, PositiveSaliency{saliency}, stream));
  SF_CUDA(cub::DeviceSelect::Flagged(nullptr, flagged_bytes, positions, static_cast<const uint8_t*>(nullptr),
                                     static_cast<int32_t*>(nullptr), static_cast<int32_t*>(nullptr), n, stream));
  // scratch: candidates int32[n] | flags uint8[n] | two counts | CUB temp, each 256-byte aligned
  auto up = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t cand_bytes = up(size_t(n) * sizeof(int32_t)), flag_bytes = up(size_t(n)), num_bytes = 256;
  const size_t temp_bytes = up(std::max(if_bytes, flagged_bytes));
  Scratch scratch(stream);
  char* base = nullptr;
  SF_CUDA(scratch.alloc(&base, cand_bytes + flag_bytes + num_bytes + temp_bytes));
  int32_t* cand = reinterpret_cast<int32_t*>(base);
  uint8_t* flags = reinterpret_cast<uint8_t*>(base + cand_bytes);
  int32_t* nums = reinterpret_cast<int32_t*>(base + cand_bytes + flag_bytes);  // [0] candidates, [1] keypoints
  void* temp = base + cand_bytes + flag_bytes + num_bytes;
  size_t bytes = temp_bytes;
  SF_CUDA(cub::DeviceSelect::If(temp, bytes, positions, cand, nums, n, PositiveSaliency{saliency}, stream));
  SF_CUDA(cudaMemsetAsync(flags, 0, size_t(n), stream));
  int blocks = 0, device = 0;
  cudaGetDevice(&device);
  cudaDeviceGetAttribute(&blocks, cudaDevAttrMultiProcessorCount, device);
  // enough warps to cover the SMs several times over; each walks the candidates with a grid stride
  const int64_t want = std::min<int64_t>(int64_t(blocks) * 8, (int64_t(n) + 7) / 8);
  iss_nms_kernel<<<unsigned(std::max<int64_t>(want, 1)), 256, 0, stream>>>(
      g->view(), saliency, cand, nums, non_max_radius * non_max_radius, min_neighbors, flags);
  SF_CUDA(cudaGetLastError());
  bytes = temp_bytes;
  SF_CUDA(cub::DeviceSelect::Flagged(temp, bytes, positions, flags, keypoints, nums + 1, n, stream));
  int32_t selected = 0;
  SF_CUDA(cudaMemcpyAsync(&selected, nums + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  *count_host = selected;
  return SF_OK;
}
