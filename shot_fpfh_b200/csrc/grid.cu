// Kernel group G: uniform-grid spatial hash with sort-by-cell, and fixed-radius search into CSR neighbour lists.
// Replaces sklearn.neighbors.KDTree(points).query_radius(queries, r) — reference call sites
// shot_parallelization.py:167-169, :220-222, :229-231, :283-285; fpfh.py:26-30; shot.py:340-341.
//
// Layout in HBM after sf_grid_build (n points, cell edge c >= 1.001 * radius):
//   pts[n]        double4  cell-sorted coordinates, .w = original index (int64 bit pattern)    32 B / point
//   nrm[n]        double4  cell-sorted normals                                                  32 B / point
//   perm[n], inv_perm[n]   int32   sorted position <-> original index
//   cell_start[ncells + 1] int32   exclusive prefix of the per-cell counts, key = (z*ny + y)*nx + x
// The predicate is sklearn's, bit for bit: ((dx*dx + dy*dy) + dz*dz) <= r*r in float64 without FMA contraction.
#include <cub/cub.cuh>
#include <stdarg.h>

#include <algorithm>
#include <cmath>

#include "sf_common.cuh"

namespace sf {

static thread_local char g_error[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

// ---- bounding box: per-block reduction + one atomic per block on the ordered-int image of the doubles -----
__device__ __forceinline__ unsigned long long ordered_bits(double v) {
  const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double from_ordered_bits(unsigned long long o) {
  const unsigned long long b = (o >> 63) ? (o & 0x7fffffffffffffffull) : ~o;
#if defined(__CUDA_ARCH__)
  return __longlong_as_double(static_cast<long long>(b));
#else
  double d;
  memcpy(&d, &b, sizeof(d));
  return d;
#endif
}

__global__ void bbox_init_kernel(unsigned long long* box) {
  if (threadIdx.x < 3) box[threadIdx.x] = ~0ull;
  else if (threadIdx.x < 6) box[threadIdx.x] = 0ull;
}

__global__ void __launch_bounds__(256) bbox_kernel(const double* __restrict__ xyz, int64_t n, unsigned long long* box) {
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double v = xyz[3 * i + a];
      lo[a] = fmin(lo[a], v);
      hi[a] = fmax(hi[a], v);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[a] = fmin(lo[a], __shfl_xor_sync(kFull, lo[a], o));
      hi[a] = fmax(hi[a], __shfl_xor_sync(kFull, hi[a], o));
    }
  }
  // warp leaders -> shared memory -> six atomics per BLOCK (one per warp serialised ~57k atomics on six words)
  __shared__ double part[8][6];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      part[warp][a] = lo[a];
      part[warp][3 + a] = hi[a];
    }
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double v = part[0][threadIdx.x];
    for (int w = 1; w < int(blockDim.x >> 5); ++w)
      v = threadIdx.x < 3 ? fmin(v, part[w][threadIdx.x]) : fmax(v, part[w][threadIdx.x]);
    if (threadIdx.x < 3) atomicMin(box + threadIdx.x, ordered_bits(v));
    else atomicMax(box + threadIdx.x, ordered_bits(v));
  }
}

// ---- cell keys + per-cell histogram ----------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    key_kernel(const double* __restrict__ xyz, int64_t n, GridView g, uint32_t* __restrict__ keys,
               int32_t* __restrict__ vals, int32_t* __restrict__ cell_count, int by_slot, int32_t* __restrict__ status) {
  // status != nullptr: a speculative build on the box of a previous one — a point outside that box (or not finite)
  // raises the flag (sf_grid_poll); the clamp keeps the build memory-safe meanwhile
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  int c[3];
  bool inside = true;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double x = xyz[3 * i + a];
    c[a] = cell_coord(x, g.origin[a], g.inv_cell, g.dims[a]);
    inside = inside && isfinite(x) && c[a] >= 0 && c[a] <= g.dims[a] - 1;
    c[a] = min(max(c[a], 0), g.dims[a] - 1);
  }
  if (status != nullptr && !inside) *status = 1;
  const uint32_t key = (uint32_t(c[2]) * g.dims[1] + c[1]) * g.dims[0] + c[0];
  keys[i] = key;
  // vals: the point's index (radix-sort path) or its arrival slot inside the cell (counting-sort path)
  const int slot = atomicAdd(cell_count + key, 1);
  vals[i] = by_slot ? slot : int32_t(i);
}

// ---- float32 side copy of a cell-sorted point (sf_math.cuh "float32-filtered decisions") ---------------------------
__device__ __forceinline__ void write_side_copy(const GridView& g, double px, double py, double pz, double nx,
                                                double ny, double nz, bool has_normal, float4* xyzc, float4* nrm32) {
  const double p[3] = {px, py, pz};
  int c[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {  // the cell key_kernel put the point in
    c[a] = cell_coord(p[a], g.origin[a], g.inv_cell, g.dims[a]);
    c[a] = min(max(c[a], 0), g.dims[a] - 1);
  }
  float l[3];
  shot_cell_local(p, g.origin, g.cell, c, l);
  *xyzc = make_float4(l[0], l[1], l[2], __uint_as_float(shot_cellbits(c)));
  if (has_normal) *nrm32 = make_float4(float(nx), float(ny), float(nz), 0.0f);
}

// ---- counting sort by cell, made stable --------------------------------------------------------------------------
// The histogram of the cells is needed anyway (cell_start), and its atomicAdd hands every point a unique slot in its
// cell: scattering to cell_start[key] + slot sorts the cloud by cell without a radix sort (three 8-bit passes over
// key-value pairs: 60 of the 127 us of kernels in the build at 1M points). The arrival order is not reproducible, so
// a second kernel RANKS each point inside its cell by original index — the count of cell-mates with a smaller index,
// read from the scattered index list (7.6 mates on average at C2 / C3) — which is exactly the order of the stable
// radix sort: the permutation, hence every result, is bit-identical to the sorted build and from run to run.
// Cost is sum over cells of population^2 / 32-ish index reads: below the 27-cell candidate scans every use of the
// grid performs afterwards, whatever the cloud.
__global__ void __launch_bounds__(256)
    place_kernel(const uint32_t* __restrict__ keys, const int32_t* __restrict__ slots, int64_t n,
                 const int32_t* __restrict__ cell_start, int2* __restrict__ arrived) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const uint32_t key = keys[i];
  arrived[cell_start[key] + slots[i]] = make_int2(int32_t(i), int32_t(key));  // (one 8-byte store: one sector)
}

// One thread per SLOT of the cell-sorted order (round 2; the first version ran one thread per point in input order:
// 32 lanes walked 32 different cells, 30 M sector look-ups for 1M points, 89 us, LSU-bound). A warp now covers 32
// neighbouring slots = about four cells: the cell bounds, the walk over the cell-mates and every store of the sorted
// arrays (a permutation inside the cell) touch the same few lines, and only the point's own coordinates and normal
// are gathered from input order.
__global__ void __launch_bounds__(256)
    rank_reorder_kernel(const double* __restrict__ xyz, const double* __restrict__ normals, int64_t n,
                        const int32_t* __restrict__ cell_start, const int2* __restrict__ arrived,
                        int32_t* __restrict__ perm, double4* __restrict__ pts, double4* __restrict__ nrm,
                        int32_t* __restrict__ inv_perm, GridView g, float4* __restrict__ xyzc,
                        float4* __restrict__ nrm32) {
  const int64_t t0 = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (t0 >= n) return;
  const int2 mine = arrived[t0];
  const int64_t i = mine.x;
  // the point's own data first: these loads are in flight while the cell-mates are counted
  const double px = __ldg(xyz + 3 * i), py = __ldg(xyz + 3 * i + 1), pz = __ldg(xyz + 3 * i + 2);
  double nx = 0.0, ny = 0.0, nz = 0.0;
  if (normals != nullptr) {
    nx = __ldg(normals + 3 * i); ny = __ldg(normals + 3 * i + 1); nz = __ldg(normals + 3 * i + 2);
  }
  const int b = cell_start[mine.y], e = cell_start[mine.y + 1];
  int rank = 0;
#pragma unroll 4
  for (int t = b; t < e; ++t) rank += arrived[t].x < mine.x;
  const int s = b + rank;
  perm[s] = mine.x;
  inv_perm[i] = s;
  pts[s] = make_double4(px, py, pz, __longlong_as_double(static_cast<long long>(i)));
  if (normals != nullptr) nrm[s] = make_double4(nx, ny, nz, 0.0);
  write_side_copy(g, px, py, pz, nx, ny, nz, normals != nullptr, xyzc + s, nrm32 + s);
}

// ---- gather into cell order ------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    reorder_kernel(const double* __restrict__ xyz, const double* __restrict__ normals, int64_t n,
                   const int32_t* __restrict__ perm, double4* __restrict__ pts, double4* __restrict__ nrm,
                   int32_t* __restrict__ inv_perm, GridView g, float4* __restrict__ xyzc, float4* __restrict__ nrm32) {
  const int64_t s = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (s >= n) return;
  const int32_t i = perm[s];
  inv_perm[i] = int32_t(s);
  const double px = xyz[3 * int64_t(i)], py = xyz[3 * int64_t(i) + 1], pz = xyz[3 * int64_t(i) + 2];
  double nx = 0.0, ny = 0.0, nz = 0.0;
  pts[s] = make_double4(px, py, pz, __longlong_as_double(static_cast<long long>(i)));
  if (normals != nullptr) {
    nx = normals[3 * int64_t(i)]; ny = normals[3 * int64_t(i) + 1]; nz = normals[3 * int64_t(i) + 2];
    nrm[s] = make_double4(nx, ny, nz, 0.0);
  }
  write_side_copy(g, px, py, pz, nx, ny, nz, normals != nullptr, xyzc + s, nrm32 + s);
}

// ---- fixed-radius search: one warp per query ---------------------------------------------------------------
// queries == nullptr means "the cloud's own points, in cell-sorted order" (the FPFH case, fpfh.py:28-30).
template <bool kFill>
__global__ void __launch_bounds__(256)
    radius_kernel(GridView g, const double* __restrict__ queries, int64_t self_first, int64_t nq, double r2,
                  int32_t* __restrict__ counts, const int64_t* __restrict__ offsets,
                  int32_t* __restrict__ nbr_sorted, int32_t* __restrict__ nbr_index, double* __restrict__ dist) {
  const int lane = threadIdx.x & 31;
  const int64_t q = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (q >= nq) return;
  double qx, qy, qz;
  if (queries != nullptr) {
    qx = __ldg(queries + 3 * q);
    qy = __ldg(queries + 3 * q + 1);
    qz = __ldg(queries + 3 * q + 2);
  } else {
    const double4 p = load_pt(g.pts + self_first + q);
    qx = p.x; qy = p.y; qz = p.z;
  }
  const Runs runs = build_runs(g, qx, qy, qz, lane, r2);  // (cells out of reach dropped)
  const int total = runs.pref[9];
  int64_t out = kFill ? offsets[q] : 0;
  int count = 0;
  for (int base = 0; base < total; base += 32) {
    const int v = base + lane;
    bool hit = false;
    int pos = 0;
    double d2 = 0.0;
    double4 p = make_double4(0, 0, 0, 0);
    if (v < total) {
      pos = run_position(runs, v);
      p = load_pt(g.pts + pos);
      d2 = rdist3(qx - p.x, qy - p.y, qz - p.z);
      hit = d2 <= r2;
    }
    const unsigned mask = __ballot_sync(kFull, hit);
    if (kFill) {
      if (hit) {
        const int64_t o = out + __popc(mask & lanemask_lt());
        if (nbr_sorted != nullptr) nbr_sorted[o] = pos;
        if (nbr_index != nullptr) nbr_index[o] = int32_t(__double_as_longlong(p.w));
        if (dist != nullptr) dist[o] = sqrt(d2);
      }
      out += __popc(mask);
    } else {
      count += __popc(mask);
    }
  }
  if (!kFill && lane == 0) counts[q] = count;
}

__global__ void widen_total_kernel(const int32_t* counts, int64_t* offsets, int64_t nq) {
  // offsets[0..nq) hold the exclusive scan; close the CSR with offsets[nq] = offsets[nq-1] + counts[nq-1].
  if (threadIdx.x == 0 && blockIdx.x == 0) offsets[nq] = nq > 0 ? offsets[nq - 1] + counts[nq - 1] : 0;
}

struct CountToI64 {
  __host__ __device__ int64_t operator()(int32_t c) const { return int64_t(c); }
};

static int ensure_temp(sf_grid* g, size_t bytes) {
  if (bytes <= g->cub_bytes) return SF_OK;
  if (g->cub_temp) SF_CUDA(cudaFree(g->cub_temp));
  g->cub_temp = nullptr;
  g->cub_bytes = 0;
  SF_CUDA(cudaMalloc(&g->cub_temp, bytes));
  g->cub_bytes = bytes;
  return SF_OK;
}

}  // namespace sf

using namespace sf;

extern "C" const char* sf_last_error(void) { return sf::g_error; }
extern "C" int sf_abi_version(void) { return SF_ABI_VERSION; }

extern "C" int sf_grid_create(sf_grid** out) {
  SF_REQUIRE(out != nullptr, SF_ERR_ARG, "sf_grid_create: null output");
  *out = new sf_grid();
  SF_CUDA(cudaGetDevice(&(*out)->device));
  return SF_OK;
}

static void free_all(sf_grid* g) {
  cudaFree(g->pts); cudaFree(g->nrm); cudaFree(g->xyzc); cudaFree(g->nrm32); cudaFree(g->perm); cudaFree(g->inv_perm);
  cudaFree(g->cell_start); cudaFree(g->cell_count); cudaFree(g->keys_in); cudaFree(g->keys_out);
  cudaFree(g->vals_in); cudaFree(g->bbox); cudaFree(g->cub_temp);
  cudaFree(g->status_dev);
  cudaFree(g->shot_cand_offsets); cudaFree(g->shot_counts); cudaFree(g->shot_lrf);
  cudaFree(g->shot_runs);
  cudaFree(g->shot_frame32); cudaFree(g->shot_worklist); cudaFree(g->shot_pairs);
  cudaFree(g->shot_nbr);
}

extern "C" int sf_grid_destroy(sf_grid* g) {
  if (g == nullptr) return SF_OK;
  free_all(g);
  delete g;
  return SF_OK;
}

static int build_cells(sf_grid* g, const double* xyz, const double* normals, int64_t n, bool check_box, cudaStream_t stream);

extern "C" int sf_grid_set_speculative(sf_grid* g, int32_t enable) {
  SF_REQUIRE(g != nullptr, SF_ERR_ARG, "sf_grid_set_speculative: null grid");
  g->speculative = enable;  // bit 0: sf_grid_build assumes the previous box; bit 1: sf_shot_single_scale the list size
  return SF_OK;
}

// The flag is read here, once, rather than copied to the host at the end of every call: a device-to-host copy between
// the kernels of a repeated step costs more than the copy itself (the stream waits for the copy engine and back).
extern "C" int sf_grid_poll(sf_grid* g, int32_t* status) {
  SF_REQUIRE(g != nullptr && status != nullptr, SF_ERR_ARG, "sf_grid_poll: null argument");
  *status = 0;
  if (g->status_dev != nullptr) SF_CUDA(cudaMemcpy(status, g->status_dev, sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (*status != 0) {  // what was assumed does not hold: the next calls read everything back again
    g->sized = false;
    g->shot_entries_per_query = 0;
    SF_CUDA(cudaMemset(g->status_dev, 0, sizeof(int32_t)));
  }
  return SF_OK;
}

// Buffers of the handle for a cloud of n points.
static int reserve_points(sf_grid* g, const double* xyz, const double* normals, int64_t n, double radius, const char* who) {
  SF_REQUIRE(g != nullptr && xyz != nullptr, SF_ERR_ARG, "%s: null grid or points", who);
  SF_REQUIRE(n > 0 && n < (int64_t(1) << 31), SF_ERR_ARG, "%s: n = %lld out of range", who, (long long)n);
  SF_REQUIRE(radius > 0.0 && std::isfinite(radius), SF_ERR_ARG, "%s: radius must be positive and finite", who);
  if (n > g->capacity) {
    cudaFree(g->pts); cudaFree(g->nrm); cudaFree(g->xyzc); cudaFree(g->nrm32); cudaFree(g->perm); cudaFree(g->inv_perm);
    cudaFree(g->keys_in); cudaFree(g->keys_out); cudaFree(g->vals_in);
    g->capacity = 0;
    SF_CUDA(cudaMalloc(&g->pts, n * sizeof(double4)));
    SF_CUDA(cudaMalloc(&g->nrm, n * sizeof(double4)));
    SF_CUDA(cudaMalloc(&g->xyzc, n * sizeof(float4)));
    SF_CUDA(cudaMalloc(&g->nrm32, n * sizeof(float4)));
    SF_CUDA(cudaMalloc(&g->perm, n * sizeof(int32_t)));
    SF_CUDA(cudaMalloc(&g->inv_perm, n * sizeof(int32_t)));
    SF_CUDA(cudaMalloc(&g->keys_in, n * sizeof(uint32_t)));
    SF_CUDA(cudaMalloc(&g->keys_out, 2 * n * sizeof(uint32_t)));  // (radix: n keys; counting sort: n int2)
    SF_CUDA(cudaMalloc(&g->vals_in, n * sizeof(int32_t)));
    g->capacity = n;
  }
  if (g->bbox == nullptr) SF_CUDA(cudaMalloc(&g->bbox, 6 * sizeof(double)));
  g->n = n;
  g->has_normals = normals != nullptr;
  if (g->status_dev == nullptr) {
    SF_CUDA(cudaMalloc(&g->status_dev, sizeof(int32_t)));
    SF_CUDA(cudaMemset(g->status_dev, 0, sizeof(int32_t)));
  }
  return SF_OK;
}

// Cell edge and table dimensions for a bounding box: the edge is slightly above the radius so that rounding in the
// cell coordinate can never push a point within `radius` of a query two cells away; grown when the dense table would
// exceed 2^25 cells.
static int grid_geometry(const double lo[3], const double hi[3], double radius, double* cell_out, int dims[3],
                         int64_t* ncells_out) {
  for (int a = 0; a < 3; ++a)
    SF_REQUIRE(std::isfinite(lo[a]) && std::isfinite(hi[a]) && hi[a] >= lo[a], SF_ERR_ARG,
               "grid geometry: non-finite coordinates or an empty box");
  double cell = radius * 1.001;
  const double kMaxCells = double(1 << 25);
  for (int iter = 0; iter < 64; ++iter) {
    double cells = 1.0;
    for (int a = 0; a < 3; ++a) cells *= std::floor((hi[a] - lo[a]) * (1.0 / cell)) + 1.0;
    if (cells <= kMaxCells) break;
    cell *= std::cbrt(cells / kMaxCells) * 1.01;
  }
  int64_t ncells = 1;
  for (int a = 0; a < 3; ++a) {
    dims[a] = int(std::floor((hi[a] - lo[a]) * (1.0 / cell))) + 1;
    ncells *= dims[a];
  }
  SF_REQUIRE(ncells <= (int64_t(1) << 26), SF_ERR_ARG, "grid geometry: %lld cells", (long long)ncells);
  *cell_out = cell;
  *ncells_out = ncells;
  return SF_OK;
}

static int adopt_geometry(sf_grid* g, const double lo[3], const double hi[3], int64_t n, double radius) {
  double cell;
  int dims[3];
  int64_t ncells;
  if (int rc = grid_geometry(lo, hi, radius, &cell, dims, &ncells)) return rc;
  g->cell = cell;
  for (int a = 0; a < 3; ++a) {
    g->origin[a] = lo[a];
    g->dims[a] = dims[a];
  }
  g->ncells = ncells;
  g->sized = true;
  g->sized_n = n;
  g->sized_radius = radius;
  g->shot_entries_per_query = 0;  // another cloud: the neighbour list is sized afresh
  return SF_OK;
}

extern "C" int sf_grid_geometry(const double* lo3, const double* hi3, double radius, double* cell, int32_t* dims3,
                                int64_t* ncells) {
  SF_REQUIRE(lo3 && hi3 && cell && dims3 && ncells && radius > 0.0, SF_ERR_ARG, "sf_grid_geometry: bad arguments");
  int dims[3];
  if (int rc = grid_geometry(lo3, hi3, radius, cell, dims, ncells)) return rc;
  for (int a = 0; a < 3; ++a) dims3[a] = dims[a];
  return SF_OK;
}

extern "C" int sf_grid_build(sf_grid* g, const double* xyz, const double* normals, int64_t n, double radius,
                             void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (int rc = reserve_points(g, xyz, normals, n, radius, "sf_grid_build")) return rc;
  // 1. bounding box (device) -> host, the only synchronisation of the build — skipped on a handle in speculative mode
  //    whose last synchronising build saw the same number of points and the same radius: the box of that build is
  //    assumed and checked on the device (sf_grid_poll tells)
  const bool assume_box = (g->speculative & 1) && g->sized && n == g->sized_n && radius == g->sized_radius;
  if (assume_box) return build_cells(g, xyz, normals, n, true, stream);  // (the key kernel checks every point)
  unsigned long long* box = reinterpret_cast<unsigned long long*>(g->bbox);
  bbox_init_kernel<<<1, 32, 0, stream>>>(box);
  const int bbox_blocks = int(std::min<int64_t>((n + 255) / 256, 148 * 4));
  bbox_kernel<<<bbox_blocks, 256, 0, stream>>>(xyz, n, box);
  unsigned long long hbox[6];
  SF_CUDA(cudaMemcpyAsync(hbox, box, sizeof(hbox), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  double lo[3], hi[3];
  for (int a = 0; a < 3; ++a) {
    lo[a] = from_ordered_bits(hbox[a]);
    hi[a] = from_ordered_bits(hbox[3 + a]);
    SF_REQUIRE(std::isfinite(lo[a]) && std::isfinite(hi[a]), SF_ERR_ARG, "sf_grid_build: non-finite coordinates");
  }
  // 2. cell edge and table dimensions
  if (int rc = adopt_geometry(g, lo, hi, n, radius)) return rc;
  return build_cells(g, xyz, normals, n, false, stream);
}

// The same build inside a box the CALLER gives (no bounding-box pass, no synchronisation): the cells are those of any
// other cloud built in that box with that radius. This is what a rank of a spatially partitioned job uses
// (shot_fpfh_b200/distributed.py, "halo"): it sorts only the points of its slab and of the cells around it, in the
// geometry of the whole cloud, and finds every neighbourhood exactly as the build of the whole cloud would lay it out.
// Every point is checked against the box on the device (sf_grid_poll reports 1 when one lies outside).
extern "C" int sf_grid_build_in_box(sf_grid* g, const double* xyz, const double* normals, int64_t n, double radius,
                                    const double* lo3, const double* hi3, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(lo3 != nullptr && hi3 != nullptr, SF_ERR_ARG, "sf_grid_build_in_box: null box");
  if (int rc = reserve_points(g, xyz, normals, n, radius, "sf_grid_build_in_box")) return rc;
  if (int rc = adopt_geometry(g, lo3, hi3, n, radius)) return rc;
  return build_cells(g, xyz, normals, n, true, stream);
}

// Steps 3-5 of the build for the geometry held by the handle.
static int build_cells(sf_grid* g, const double* xyz, const double* normals, int64_t n, bool check_box, cudaStream_t stream) {
  const int64_t ncells = g->ncells;
  if (ncells + 1 > g->cells_capacity) {
    cudaFree(g->cell_start); cudaFree(g->cell_count);
    g->cells_capacity = 0;
    SF_CUDA(cudaMalloc(&g->cell_start, (ncells + 1) * sizeof(int32_t)));
    SF_CUDA(cudaMalloc(&g->cell_count, (ncells + 1) * sizeof(int32_t)));
    g->cells_capacity = ncells + 1;
  }
  // 3. keys + histogram, 4. prefix over cells, 5. sort by cell (stable: ascending original index inside a cell) and
  // gather into cell order: counting sort + rank (see place_kernel); SF_GRID_RADIX=1 keeps the CUB radix sort of
  // (key, index) pairs, which gives the same permutation (tests compare the two)
  SF_CUDA(cudaMemsetAsync(g->cell_count, 0, (ncells + 1) * sizeof(int32_t), stream));
  const GridView view = g->view();
  const int blocks = int((n + 255) / 256);
  const char* radix_env = getenv("SF_GRID_RADIX");
  const bool radix = radix_env != nullptr && radix_env[0] == '1';
  key_kernel<<<blocks, 256, 0, stream>>>(xyz, n, view, g->keys_in, g->vals_in, g->cell_count, radix ? 0 : 1,
                                         check_box ? g->status_dev : nullptr);
  int end_bit = 1;
  while ((int64_t(1) << end_bit) < ncells) ++end_bit;
  size_t sort_bytes = 0, scan_bytes = 0;
  if (radix)
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, g->keys_in, g->keys_out, g->vals_in, g->perm, int(n), 0,
                                    end_bit, stream);
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, g->cell_count, g->cell_start, int(ncells + 1), stream);
  if (int rc = ensure_temp(g, std::max(sort_bytes, scan_bytes) + 256)) return rc;
  size_t bytes = g->cub_bytes;
  if (radix) {
    SF_CUDA(cub::DeviceRadixSort::SortPairs(g->cub_temp, bytes, g->keys_in, g->keys_out, g->vals_in, g->perm, int(n), 0,
                                            end_bit, stream));
    bytes = g->cub_bytes;
  }
  SF_CUDA(cub::DeviceScan::ExclusiveSum(g->cub_temp, bytes, g->cell_count, g->cell_start, int(ncells + 1), stream));
  if (radix) {
    reorder_kernel<<<blocks, 256, 0, stream>>>(xyz, normals, n, g->perm, g->pts, g->nrm, g->inv_perm, view, g->xyzc,
                                               g->nrm32);
  } else {
    int2* arrived = reinterpret_cast<int2*>(g->keys_out);  // (index, cell) per slot of the arrival order
    place_kernel<<<blocks, 256, 0, stream>>>(g->keys_in, g->vals_in, n, g->cell_start, arrived);
    rank_reorder_kernel<<<blocks, 256, 0, stream>>>(xyz, normals, n, g->cell_start, arrived, g->perm, g->pts, g->nrm,
                                                    g->inv_perm, view, g->xyzc, g->nrm32);
  }
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_grid_info(const sf_grid* g, int64_t* n, int64_t* ncells, double* cell, int32_t* dims3) {
  SF_REQUIRE(g != nullptr, SF_ERR_ARG, "sf_grid_info: null grid");
  if (n) *n = g->n;
  if (ncells) *ncells = g->ncells;
  if (cell) *cell = g->cell;
  if (dims3) for (int a = 0; a < 3; ++a) dims3[a] = g->dims[a];
  return SF_OK;
}

extern "C" int sf_grid_permutation(const sf_grid* g, int32_t* perm_out, int32_t* inv_perm_out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_grid_permutation: grid not built");
  if (perm_out)
    SF_CUDA(cudaMemcpyAsync(perm_out, g->perm, g->n * sizeof(int32_t), cudaMemcpyDeviceToDevice, stream));
  if (inv_perm_out)
    SF_CUDA(cudaMemcpyAsync(inv_perm_out, g->inv_perm, g->n * sizeof(int32_t), cudaMemcpyDeviceToDevice, stream));
  return SF_OK;
}

extern "C" int sf_grid_arrays(const sf_grid* g, double* pts_out, double* nrm_out, float* xyzc_out, float* nrm32_out,
                              int32_t* cell_start_out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_grid_arrays: grid not built");
  SF_REQUIRE(g->has_normals || (nrm_out == nullptr && nrm32_out == nullptr), SF_ERR_ARG,
             "sf_grid_arrays: the grid was built without normals");
  const auto copy = [&](void* dst, const void* src, size_t bytes) {
    return dst != nullptr ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, stream) : cudaSuccess;
  };
  SF_CUDA(copy(pts_out, g->pts, g->n * sizeof(double4)));
  SF_CUDA(copy(nrm_out, g->nrm, g->n * sizeof(double4)));
  SF_CUDA(copy(xyzc_out, g->xyzc, g->n * sizeof(float4)));
  SF_CUDA(copy(nrm32_out, g->nrm32, g->n * sizeof(float4)));
  SF_CUDA(copy(cell_start_out, g->cell_start, (g->ncells + 1) * sizeof(int32_t)));
  return SF_OK;
}

extern "C" int sf_radius_count(sf_grid* g, const double* queries, int64_t self_first, int64_t nq, double radius,
                               int64_t* offsets,
                               int64_t* total_host, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_radius_count: grid not built");
  SF_REQUIRE(offsets != nullptr && nq >= 0, SF_ERR_ARG, "sf_radius_count: bad arguments");
  SF_REQUIRE(radius_fits(g, radius), SF_ERR_ARG,
             "sf_radius_count: radius %g exceeds the cell edge %g the grid was built for", radius, g->cell);
  if (queries == nullptr)
    SF_REQUIRE(self_first >= 0 && self_first + nq <= g->n, SF_ERR_ARG, "self-query range [%lld, %lld) outside the cloud",
               (long long)self_first, (long long)(self_first + nq));
  if (nq == 0) {
    SF_CUDA(cudaMemsetAsync(offsets, 0, sizeof(int64_t), stream));
    if (total_host) *total_host = 0;
    return SF_OK;
  }
  // counts live in the (now free) sort scratch when it is large enough, else in a fresh temp
  size_t scan_bytes = 0;
  cub::TransformInputIterator<int64_t, CountToI64, const int32_t*> dummy(nullptr, CountToI64());
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, dummy, offsets, int(nq), stream);
  const size_t counts_bytes = ((size_t(nq) * sizeof(int32_t) + 255) / 256) * 256;
  if (int rc = ensure_temp(g, counts_bytes + scan_bytes + 256)) return rc;
  int32_t* counts = static_cast<int32_t*>(g->cub_temp);
  void* scan_temp = static_cast<char*>(g->cub_temp) + counts_bytes;
  const double r2 = radius * radius;
  const int64_t threads = nq * 32;
  radius_kernel<false><<<unsigned((threads + 255) / 256), 256, 0, stream>>>(g->view(), queries, self_first, nq, r2, counts,
                                                                           nullptr, nullptr, nullptr, nullptr);
  cub::TransformInputIterator<int64_t, CountToI64, const int32_t*> in(counts, CountToI64());
  size_t bytes = scan_bytes + 256;
  SF_CUDA(cub::DeviceScan::ExclusiveSum(scan_temp, bytes, in, offsets, int(nq), stream));
  widen_total_kernel<<<1, 32, 0, stream>>>(counts, offsets, nq);
  SF_CUDA(cudaGetLastError());
  if (total_host != nullptr) {
    SF_CUDA(cudaMemcpyAsync(total_host, offsets + nq, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
    SF_CUDA(cudaStreamSynchronize(stream));
  }
  return SF_OK;
}

extern "C" int sf_radius_fill(sf_grid* g, const double* queries, int64_t self_first, int64_t nq, double radius,
                              const int64_t* offsets,
                              int32_t* nbr_sorted, int32_t* nbr_index, double* dist, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_radius_fill: grid not built");
  SF_REQUIRE(offsets != nullptr && nq >= 0, SF_ERR_ARG, "sf_radius_fill: bad arguments");
  SF_REQUIRE(radius_fits(g, radius), SF_ERR_ARG, "sf_radius_fill: radius exceeds the cell edge");
  if (queries == nullptr)
    SF_REQUIRE(self_first >= 0 && self_first + nq <= g->n, SF_ERR_ARG, "self-query range [%lld, %lld) outside the cloud",
               (long long)self_first, (long long)(self_first + nq));
  if (nq == 0) return SF_OK;
  const int64_t threads = nq * 32;
  radius_kernel<true><<<unsigned((threads + 255) / 256), 256, 0, stream>>>(
      g->view(), queries, self_first, nq, radius * radius, nullptr, offsets, nbr_sorted, nbr_index, dist);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}
