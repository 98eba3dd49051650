// Result transport, device side: dense float32 rows -> compact rows (per-row offsets, uint16 columns, float32 values
// of the non-zero entries, in row order and ascending column order). See host_io.cpp for why: the (Q, 352) float64
// array the reference API returns is ~86 % zeros and its device->host copy is what bounds the end-to-end call.
#include <cub/cub.cuh>

#include "sf_common.cuh"

namespace sf {

// One warp per row; lane l looks at columns l, l + 32, ... (coalesced), so the entries of round j precede those of
// round j + 1 and, inside a round, lane order is column order.
template <bool kFill>
__global__ void __launch_bounds__(256)
    compact_rows_kernel(const float* __restrict__ dense, int64_t n_rows, int width, int64_t* __restrict__ counts,
                        const int64_t* __restrict__ offsets, uint16_t* __restrict__ cols, float* __restrict__ vals) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (r >= n_rows) return;
  const float* row = dense + r * width;
  int64_t out = kFill ? offsets[r] : 0;
  int count = 0;
  for (int base = 0; base < width; base += 32) {
    const int c = base + lane;
    const float v = c < width ? __ldg(row + c) : 0.0f;
    const bool keep = v != 0.0f;
    const unsigned mask = __ballot_sync(kFull, keep);
    if (kFill) {
      if (keep) {
        const int64_t o = out + __popc(mask & lanemask_lt());
        cols[o] = uint16_t(c);
        vals[o] = v;
      }
      out += __popc(mask);
    } else {
      count += __popc(mask);
    }
  }
  if (!kFill && lane == 0) counts[r] = count;
}

}  // namespace sf

using namespace sf;

// offsets_dev: int64 (n_rows + 1), exclusive prefix of the per-row non-zero counts; *total_host = offsets[n_rows]
// (synchronises `stream`). scratch: offsets_dev doubles as the count buffer, the scan runs in place.
extern "C" int sf_rows_compact_count(const float* dense, int64_t n_rows, int32_t width, int64_t* offsets_dev,
                                     int64_t* total_host, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(n_rows >= 0 && width > 0 && width <= 65536 && offsets_dev && total_host, SF_ERR_ARG,
             "sf_rows_compact_count: bad arguments");
  SF_REQUIRE(n_rows == 0 || dense != nullptr, SF_ERR_ARG, "sf_rows_compact_count: null rows");
  SF_REQUIRE(n_rows < (int64_t(1) << 31) - 1, SF_ERR_CAPACITY, "sf_rows_compact_count: too many rows");
  *total_host = 0;
  SF_CUDA(cudaMemsetAsync(offsets_dev + n_rows, 0, sizeof(int64_t), stream));
  if (n_rows > 0)
    compact_rows_kernel<false><<<unsigned((n_rows * 32 + 255) / 256), 256, 0, stream>>>(dense, n_rows, width, offsets_dev,
                                                                                      nullptr, nullptr, nullptr);
  void* temp = nullptr;
  size_t temp_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, offsets_dev, offsets_dev, int(n_rows + 1), stream);
  Scratch scratch(stream);
  SF_CUDA(scratch.alloc(&temp, temp_bytes + 16));
  SF_CUDA(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, offsets_dev, offsets_dev, int(n_rows + 1), stream));
  SF_CUDA(cudaMemcpyAsync(total_host, offsets_dev + n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  return SF_OK;
}

extern "C" int sf_rows_compact_fill(const float* dense, int64_t n_rows, int32_t width, const int64_t* offsets_dev,
                                    uint16_t* cols_dev, float* vals_dev, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(n_rows >= 0 && width > 0 && width <= 65536 && offsets_dev, SF_ERR_ARG, "sf_rows_compact_fill: bad arguments");
  if (n_rows == 0) return SF_OK;
  SF_REQUIRE(dense && cols_dev && vals_dev, SF_ERR_ARG, "sf_rows_compact_fill: null buffers");
  compact_rows_kernel<true><<<unsigned((n_rows * 32 + 255) / 256), 256, 0, stream>>>(
      dense, n_rows, width, nullptr, offsets_dev, cols_dev, vals_dev);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}
