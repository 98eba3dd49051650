// Voxel-grid subsampling on the device: the support reducer that sits immediately upstream of the SHOT path
// (`grid_subsampling`, core/subsampling.py:5-39, called at shot_parallelization.py:157-161, :210-214, :273-277 when
// the pipeline passes `subsampling_voxel_size`). SURVEY.md §8f ranks it as the first "next" row: on the host it is a
// Python loop over voxels (4.4 s at 1M points) that would dominate the end-to-end time once descriptors take ms.
//
// Semantics reproduced: voxel key = np.floor_divide(p - min, voxel) per axis (NumPy's float floor division, see
// floor_divide_np), voxels in lexicographic (x, y, z) key order — what np.unique(axis=0) returns —, and per voxel
// the index of the point closest to the voxel's barycentre, first one on ties, members taken in ascending index
// order. (The reference walks the members in the order of an unstable argsort, so on exact distance ties — every
// 2-point voxel is one, up to rounding — its pick is implementation-dependent; see tests.)
#include <cub/cub.cuh>

#include "sf_common.cuh"

namespace sf {

// np.floor_divide for float64 (numpy/core/src/npymath: npy_divmod), b > 0.
__device__ __forceinline__ double floor_divide_np(double a, double b) {
  double mod = fmod(a, b);
  double div = (a - mod) / b;
  if (mod != 0.0 && mod < 0.0) div -= 1.0;  // (b < 0) != (mod < 0) with b > 0
  if (div != 0.0) {
    double fl = floor(div);
    if (div - fl > 0.5) fl += 1.0;
    return fl;
  }
  return copysign(0.0, a / b);
}

__device__ __forceinline__ double decode_ordered(unsigned long long o) {
  const unsigned long long b = (o >> 63) ? (o & 0x7fffffffffffffffull) : ~o;
  return __longlong_as_double(static_cast<long long>(b));
}
__device__ __forceinline__ unsigned long long encode_ordered(double v) {
  const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__global__ void voxel_min_init_kernel(unsigned long long* lo) {
  if (threadIdx.x < 3) lo[threadIdx.x] = ~0ull;
}

__global__ void __launch_bounds__(256) voxel_min_kernel(const double* __restrict__ xyz, int64_t n, unsigned long long* lo) {
  double m[3] = {INFINITY, INFINITY, INFINITY};
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
#pragma unroll
    for (int a = 0; a < 3; ++a) m[a] = fmin(m[a], xyz[3 * i + a]);
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m[a] = fmin(m[a], __shfl_xor_sync(kFull, m[a], o));
  }
  __shared__ double block_min[8][3];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) for (int a = 0; a < 3; ++a) block_min[warp][a] = m[a];
  __syncthreads();
  if (threadIdx.x < 3) {
    double v = block_min[0][threadIdx.x];
    for (int w = 1; w < int(blockDim.x >> 5); ++w) v = fmin(v, block_min[w][threadIdx.x]);
    atomicMin(lo + threadIdx.x, encode_ordered(v));
  }
}

// 21 bits per axis, x most significant: unsigned order of the packed key == lexicographic (kx, ky, kz) order.
__global__ void __launch_bounds__(256)
    voxel_key_kernel(const double* __restrict__ xyz, int64_t n, double voxel, const unsigned long long* __restrict__ lo,
                     unsigned long long* __restrict__ keys, int32_t* __restrict__ vals, int* __restrict__ overflow) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  unsigned long long key = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double k = floor_divide_np(xyz[3 * i + a] - decode_ordered(lo[a]), voxel);
    if (!(k >= 0.0 && k < 2097152.0)) { atomicExch(overflow, 1); }
    key = (key << 21) | static_cast<unsigned long long>(k >= 0.0 && k < 2097152.0 ? k : 0.0);
  }
  keys[i] = key;
  vals[i] = int32_t(i);
}

// One thread per voxel (the thread at the first sorted position of the voxel walks its members).
__global__ void __launch_bounds__(256)
    voxel_pick_kernel(const double* __restrict__ xyz, int64_t n, const unsigned long long* __restrict__ keys,
                      const int32_t* __restrict__ order, const int32_t* __restrict__ rank, int32_t* __restrict__ picked,
                      int32_t* __restrict__ members) {
  const int64_t s = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (s >= n) return;
  const unsigned long long key = keys[s];
  if (s > 0 && keys[s - 1] == key) return;
  double sum[3] = {0.0, 0.0, 0.0};
  int64_t e = s;
  for (; e < n && keys[e] == key; ++e) {
    const int64_t i = order[e];
#pragma unroll
    for (int a = 0; a < 3; ++a) sum[a] += xyz[3 * i + a];
  }
  const double m = double(e - s);
  const double cx = sum[0] / m, cy = sum[1] / m, cz = sum[2] / m;
  double best = INFINITY;
  int32_t best_i = -1;
  for (int64_t t = s; t < e; ++t) {
    const int64_t i = order[t];
    const double d = sqrt(rdist3(xyz[3 * i] - cx, xyz[3 * i + 1] - cy, xyz[3 * i + 2] - cz));
    if (d < best) { best = d; best_i = int32_t(i); }
  }
  picked[rank[s]] = best_i;
  if (members != nullptr) members[rank[s]] = int32_t(e - s);
}

__global__ void __launch_bounds__(256)
    voxel_flag_kernel(const unsigned long long* __restrict__ keys, int64_t n, int32_t* __restrict__ flags) {
  const int64_t s = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (s < n) flags[s] = (s == 0 || keys[s - 1] != keys[s]) ? 1 : 0;
}

}  // namespace sf

using namespace sf;

extern "C" int sf_voxel_subsample(const double* xyz, int64_t n, double voxel, int32_t* picked, int32_t* members,
                                  int64_t* count_host, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(xyz && picked && count_host && n >= 0, SF_ERR_ARG, "sf_voxel_subsample: bad arguments");
  SF_REQUIRE(voxel > 0.0 && n < (int64_t(1) << 31), SF_ERR_ARG, "sf_voxel_subsample: voxel must be > 0, n < 2^31");
  *count_host = 0;
  if (n == 0) return SF_OK;
  unsigned long long *lo = nullptr, *keys_in = nullptr, *keys_out = nullptr;
  int32_t *vals_in = nullptr, *order = nullptr, *flags = nullptr, *rank = nullptr;
  int* overflow = nullptr;
  void* temp = nullptr;
  size_t sort_bytes = 0, scan_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, keys_in, keys_out, vals_in, order, int(n), 0, 63, stream);
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, flags, rank, int(n), stream);
  const size_t temp_bytes = (sort_bytes > scan_bytes ? sort_bytes : scan_bytes) + 256;
  Scratch scratch(stream);
  SF_CUDA(scratch.alloc(&lo, 4 * sizeof(unsigned long long)));
  SF_CUDA(scratch.alloc(&keys_in, size_t(n) * 8));
  SF_CUDA(scratch.alloc(&keys_out, size_t(n) * 8));
  SF_CUDA(scratch.alloc(&vals_in, size_t(n) * 4));
  SF_CUDA(scratch.alloc(&order, size_t(n) * 4));
  SF_CUDA(scratch.alloc(&flags, size_t(n) * 4));
  SF_CUDA(scratch.alloc(&rank, size_t(n + 1) * 4));
  SF_CUDA(scratch.alloc(&overflow, sizeof(int)));
  SF_CUDA(scratch.alloc(&temp, temp_bytes));
  SF_CUDA(cudaMemsetAsync(overflow, 0, sizeof(int), stream));
  const unsigned blocks = unsigned((n + 255) / 256);
  voxel_min_init_kernel<<<1, 32, 0, stream>>>(lo);
  voxel_min_kernel<<<blocks < 1184u ? blocks : 1184u, 256, 0, stream>>>(xyz, n, lo);
  voxel_key_kernel<<<blocks, 256, 0, stream>>>(xyz, n, voxel, lo, keys_in, vals_in, overflow);
  size_t bytes = temp_bytes;
  SF_CUDA(cub::DeviceRadixSort::SortPairs(temp, bytes, keys_in, keys_out, vals_in, order, int(n), 0, 63, stream));
  voxel_flag_kernel<<<blocks, 256, 0, stream>>>(keys_out, n, flags);
  bytes = temp_bytes;
  SF_CUDA(cub::DeviceScan::ExclusiveSum(temp, bytes, flags, rank, int(n), stream));
  voxel_pick_kernel<<<blocks, 256, 0, stream>>>(xyz, n, keys_out, order, rank, picked, members);
  int32_t last_rank = 0, last_flag = 0;
  int overflow_host = 0;
  SF_CUDA(cudaMemcpyAsync(&last_rank, rank + (n - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaMemcpyAsync(&last_flag, flags + (n - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaMemcpyAsync(&overflow_host, overflow, sizeof(int), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  SF_REQUIRE(overflow_host == 0, SF_ERR_CAPACITY, "sf_voxel_subsample: more than 2^21 voxels along an axis");
  *count_host = int64_t(last_rank) + last_flag;
  return SF_OK;
}
