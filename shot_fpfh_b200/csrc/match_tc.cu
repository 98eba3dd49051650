// Kernel M1 (tensor cores): shortlist of the k nearest target rows per query row WITHOUT materialising the
// (Qa, Qb) distance matrix that the reference builds with scipy cdist (matching.py:47, :164).
//
//   score(i, j) = |b_j|^2 - 2 a_i . b_j            (|a_i|^2 is constant per row and irrelevant to the ranking)
//
// a_i . b_j is a float16 x float16 -> float32 GEMM on the 5th-generation tensor cores (tcgen05.mma kind::f16,
// accumulators in TMEM). One CTA owns 128 query rows: their operand tile A (128 x K, <= 96 KB) is loaded ONCE by
// TMA and stays resident in shared memory; the target rows stream through a 3-stage TMA pipeline in tiles of
// 256 rows x 64 columns (128-byte swizzle). Each 128 x 256 accumulator tile lives in one half of TMEM (256 of
// 512 columns) while the other half is drained by the epilogue, so the MMA of tile t+1 overlaps the top-k scan of
// tile t. The epilogue reads the accumulators with tcgen05.ld (one TMEM lane = one query row per thread), and
// keeps a per-row running top-k in registers; only (Qa, k) scores/indices ever reach HBM.
//
// Warp roles (384 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warp 2 = TMEM
// allocator, warps 4..11 = epilogue: warp w touches TMEM lanes 32*(w%4) .. +31 (a hardware restriction) and the
// column half (w-4)/4 of each tile. Its fast path is branch-free (score = fma, group minimum, one flag bit per group
// of 8 columns); the rare insertions run through ONE out-of-line loop that re-reads the flagged groups from TMEM.
// Grid: (number of 128-row query tiles, number of target splits); each split scans a contiguous range of target
// tiles; the per-split, per-half shortlists are merged by topk_merge_kernel (match.cu). Splitting keeps all 148 SMs
// busy when there are few query tiles.
//
// Round-1 measurements on B200 (200k x 200k x 352, profiles/r01_summary.md): TMA + MMA alone sustain 1.43 PFLOP/s
// (89 % of the measured cuBLAS bf16 peak), the full kernel 1.29 PFLOP/s (81 %).
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>

#include "sf_common.cuh"

namespace sf {

int launch_merge_partials(const float* score, const int32_t* idx, int parts, int64_t qa, int k, float* score_out,
                          int32_t* idx_out, cudaStream_t stream);  // match.cu

namespace tc {

constexpr int kBM = 128;        // query rows per CTA (= TMEM lanes)
constexpr int kBN = 256;        // target rows per accumulator tile (= TMEM columns per accumulator)
constexpr int kBK = 64;         // halves per K block: 128 bytes = one swizzle-128B row
constexpr int kStages = 3;      // B pipeline depth
constexpr int kMaxKBlocks = 6;  // K <= 384 (SHOT: 352 padded to 384)
// (4 parts = 16 epilogue warps were measured: 22.5 ms against 21.6 ms with 8 at 200k x 200k — 96 registers per thread
// and twice the partial lists cost more than the extra warps hide)
#ifndef SF_TC_EPI_PARTS
#define SF_TC_EPI_PARTS 2
#endif
constexpr int kEpiParts = SF_TC_EPI_PARTS;       // column parts of an accumulator tile, one epilogue warp per (lane quarter, part)
constexpr int kEpiCols = kBN / kEpiParts;        // columns per epilogue warp: 128 or 64
constexpr int kEpiChunks = kEpiCols / 32;        // TMEM loads of 32 columns per warp and tile
constexpr int kThreads = (4 + 4 * kEpiParts) * 32;  // 4 control warps + 8 or 16 epilogue warps
constexpr uint32_t kABlockBytes = kBM * kBK * 2;  // 16 KB
constexpr uint32_t kBStageBytes = kBN * kBK * 2;  // 32 KB
constexpr uint32_t kSmemA = 0;
constexpr uint32_t kSmemB = kMaxKBlocks * kABlockBytes;            // 96 KB
constexpr uint32_t kSmemBar = kSmemB + kStages * kBStageBytes;     // 192 KB
constexpr uint32_t kSmemBnorm = 4 * kEpiParts * 2 * (kEpiCols / 4) * 16;  // per epilogue warp: 2 buffers of kEpiCols floats
constexpr uint32_t kSmemBytes = kSmemBar + 256 + kSmemBnorm + 1024;  // barriers + |b|^2 staging + alignment slack

// ---- PTX wrappers -----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
// Same wait with a back-off, for the two single-thread roles (TMA producer, MMA issuer): they share a scheduler
// with an epilogue warp each, and a tight try_wait loop would steal its issue slots (ncu: 37 M spins per launch).
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
  uint32_t done;
  while (true) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(64);
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, both operands K-major, float16 in / float32 out.
__device__ __forceinline__ void tcgen05_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, "
      "%24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 8 consecutive columns of this warp's 32 lanes, loaded and waited for (slow path only).
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor of a K-major tile stored as rows of 128 bytes with the 128-byte swizzle:
// start address >> 4 in bits [0,14), leading byte offset (unused for swizzled K-major) = 1 in [16,30),
// stride byte offset = 1024 B (8 rows x 128 B) >> 4 = 64 in [32,46), descriptor version 1 in [46,48),
// layout type SWIZZLE_128B = 2 in [61,64).
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  return uint64_t((smem_addr >> 4) & 0x3FFF) | (uint64_t(1) << 16) | (uint64_t(64) << 32) | (uint64_t(1) << 46) |
         (uint64_t(2) << 61);
}
// Instruction descriptor, kind::f16: D = F32 (bits [4,6) = 1), A = B = F16 (0), K-major both, N >> 3 in [17,23),
// M >> 4 in [24,29).
constexpr uint32_t kIdesc = (1u << 4) | (uint32_t(kBN >> 3) << 17) | (uint32_t(kBM >> 4) << 24);

template <int K>
struct TopK {
  float s[K];
  int i[K];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int k = 0; k < K; ++k) { s[k] = INFINITY; i[k] = -1; }
  }
  // targets are scanned in ascending index order, so a strict `<` keeps the lowest index among equal scores
  __device__ __forceinline__ void push(float score, int index) {
    s[K - 1] = score; i[K - 1] = index;
#pragma unroll
    for (int k = K - 1; k > 0; --k) {
      if (s[k] < s[k - 1]) {
        const float ts = s[k]; s[k] = s[k - 1]; s[k - 1] = ts;
        const int ti = i[k]; i[k] = i[k - 1]; i[k - 1] = ti;
      }
    }
  }
};

template <int K>
__global__ void __launch_bounds__(kThreads, 1)
    topk_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                   const float* __restrict__ bnorm, int64_t qa, int64_t qb, int num_kb, int tiles_per_split,
                   int index_offset, float* __restrict__ score, int32_t* __restrict__ idx, int debug) {
  // `debug` (env SF_TC_DEBUG, profiling only; results are garbage when set): 1 = skip the MMAs, 2 = skip the
  // epilogue's TMEM reads / top-k, 4 = skip the B loads. Used to attribute time to TMA / MMA / epilogue.
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // swizzle-128B tiles need 1024-byte alignment
  const uint32_t bar_base = smem_base + kSmemBar;
  const uint32_t bar_a_full = bar_base;
  auto bar_b_full = [&](int s) { return bar_base + 8u * (1 + s); };
  auto bar_b_empty = [&](int s) { return bar_base + 8u * (1 + kStages + s); };
  auto bar_t_full = [&](int a) { return bar_base + 8u * (1 + 2 * kStages + a); };
  auto bar_t_empty = [&](int a) { return bar_base + 8u * (3 + 2 * kStages + a); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_raw + (bar_base - smem_u32(smem_raw)) + 8u * (5 + 2 * kStages));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * kBM;
  const int total_tiles = int((qb + kBN - 1) / kBN);
  const int tile_begin = blockIdx.y * tiles_per_split;
  const int tile_end = min(tile_begin + tiles_per_split, total_tiles);
  const int my_tiles = max(tile_end - tile_begin, 0);

  if (warp == 1 && lane == 0) {
    mbar_init(bar_a_full, 1);
    for (int s = 0; s < kStages; ++s) { mbar_init(bar_b_full(s), 1); mbar_init(bar_b_empty(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(bar_t_full(a), 1); mbar_init(bar_t_empty(a), 4 * kEpiParts * 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {  // TMEM: all 512 columns (two 128 x 256 float32 accumulators)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    // ===== TMA producer =====
    mbar_expect_tx(bar_a_full, uint32_t(num_kb) * kABlockBytes);
    for (int kb = 0; kb < num_kb; ++kb) tma_load_2d(smem_base + kSmemA + kb * kABlockBytes, &map_a, bar_a_full, kb * kBK, m0);
    int it = 0;
    for (int t = 0; t < my_tiles; ++t) {
      const int n0 = (tile_begin + t) * kBN;
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const int s = it % kStages;
        const uint32_t phase = (it / kStages) & 1;
        mbar_wait_relaxed(bar_b_empty(s), phase ^ 1);
        if (debug & 4) { mbar_arrive(bar_b_full(s)); continue; }
        mbar_expect_tx(bar_b_full(s), kBStageBytes);
        tma_load_2d(smem_base + kSmemB + s * kBStageBytes, &map_b, bar_b_full(s), kb * kBK, n0);
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===== MMA issuer =====
    mbar_wait(bar_a_full, 0);
    int it = 0;
    for (int t = 0; t < my_tiles; ++t) {
      const int acc = t & 1;
      mbar_wait_relaxed(bar_t_empty(acc), ((t >> 1) & 1) ^ 1);
      tcgen05_fence_after();
      const uint32_t tmem_d = tmem_base + uint32_t(acc * kBN);
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const int s = it % kStages;
        mbar_wait_relaxed(bar_b_full(s), (it / kStages) & 1);
        tcgen05_fence_after();
        if (debug & 1) { mbar_arrive(bar_b_empty(s)); continue; }
        const uint64_t da = make_desc(smem_base + kSmemA + kb * kABlockBytes);
        const uint64_t db = make_desc(smem_base + kSmemB + s * kBStageBytes);
#pragma unroll
        for (int k = 0; k < kBK / 16; ++k)  // UMMA_K = 16 halves = 32 bytes: +2 in the (>> 4) start-address field
          tcgen05_mma_f16(tmem_d, da + uint64_t(2 * k), db + uint64_t(2 * k), kIdesc, uint32_t((kb | k) != 0));
        tcgen05_commit(bar_b_empty(s));  // frees the B stage once the MMAs that read it have retired
      }
      if (debug & 1) mbar_arrive(bar_t_full(acc));
      else tcgen05_commit(bar_t_full(acc));  // accumulator tile complete
    }
  } else if (warp >= 4) {
    // ===== epilogue: 8 warps. Warp w reads TMEM lanes 32*(w%4).. (one query row per thread) and the column half
    // (w-4)/4 of every accumulator tile, i.e. 4 chunks of 32 columns; the two halves of a row keep separate
    // top-k lists that the merge kernel joins. Latency hiding (ncu round 1: the epilogue was pure exposed latency):
    //   - |b|^2 of the NEXT tile is fetched into a register during the current tile and parked in shared memory,
    //     so the inner loop reads it with broadcast LDS instead of waiting on L2;
    //   - the TMEM load of chunk c+1 is in flight while chunk c is processed.
    const int quarter = warp & 3;
    const int half = (warp - 4) >> 2;  // (the column part of this warp: 0 .. kEpiParts - 1)
    const int row = m0 + quarter * 32 + lane;
    constexpr int kBnVec = kEpiCols / 4;  // float4 per buffer
    float4* bn_buf = reinterpret_cast<float4*>(smem_raw + (bar_base - smem_u32(smem_raw)) + 256) + (warp - 4) * 2 * kBnVec;
    const bool bn_aligned = (reinterpret_cast<uintptr_t>(bnorm) & 15) == 0;
    auto load_bn = [&](int tile) -> float4 {  // |b|^2 of columns 4*lane .. +3 of this warp's part; +inf past the end
      if (lane >= kBnVec) return make_float4(0, 0, 0, 0);
      const int64_t col = int64_t(tile) * kBN + half * kEpiCols + 4 * lane;
      if (bn_aligned && col + 4 <= qb) return __ldg(reinterpret_cast<const float4*>(bnorm + col));
      float4 r;
      r.x = col + 0 < qb ? __ldg(bnorm + col + 0) : INFINITY;
      r.y = col + 1 < qb ? __ldg(bnorm + col + 1) : INFINITY;
      r.z = col + 2 < qb ? __ldg(bnorm + col + 2) : INFINITY;
      r.w = col + 3 < qb ? __ldg(bnorm + col + 3) : INFINITY;
      return r;
    };
    TopK<K> top;
    top.init();
    float thr = INFINITY;
    float4 bn_next = my_tiles > 0 ? load_bn(tile_begin) : make_float4(0, 0, 0, 0);
    for (int t = 0; t < my_tiles; ++t) {
      const int acc = t & 1;
      const int n0 = (tile_begin + t) * kBN + half * kEpiCols;
      float4* bn = bn_buf + acc * kBnVec;
      if (lane < kBnVec) bn[lane] = bn_next;
      __syncwarp();
      if (t + 1 < my_tiles) bn_next = load_bn(tile_begin + t + 1);
      mbar_wait(bar_t_full(acc), (t >> 1) & 1);
      tcgen05_fence_after();
      if (debug & 2) { mbar_arrive(bar_t_empty(acc)); continue; }
      const uint32_t taddr = tmem_base + (uint32_t(quarter * 32) << 16) + uint32_t(acc * kBN + half * kEpiCols);
      uint32_t va[32], vb[32];
      tmem_ld32_issue(taddr, va);
      // Pass 1, branch-free and fully unrolled: the minimum score of each group of 8 columns against the row's
      // current k-th best -> one flag bit per group (16 groups in this warp's 128 columns).
      // (ncu round 1: with the insertion code inlined at all 16 unrolled sites the kernel was 150 KB of SASS and
      // every insertion missed the instruction cache, ~4 k cycles each: 74 ms instead of 20 ms at 200k x 200k.)
      uint32_t flags = 0;
#pragma unroll
      for (int c = 0; c < kEpiChunks; ++c) {
        tmem_ld_wait();
        uint32_t(&v)[32] = (c & 1) ? vb : va;
        if (c + 1 < kEpiChunks) tmem_ld32_issue(taddr + 32 * (c + 1), (c & 1) ? va : vb);
        if (debug & 8) continue;
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) {
          const float4 b0 = bn[8 * c + 2 * g8], b1 = bn[8 * c + 2 * g8 + 1];  // same address in every lane: broadcast
          const float s0 = fmaf(-2.0f, __uint_as_float(v[8 * g8 + 0]), b0.x), s1 = fmaf(-2.0f, __uint_as_float(v[8 * g8 + 1]), b0.y);
          const float s2 = fmaf(-2.0f, __uint_as_float(v[8 * g8 + 2]), b0.z), s3 = fmaf(-2.0f, __uint_as_float(v[8 * g8 + 3]), b0.w);
          const float s4 = fmaf(-2.0f, __uint_as_float(v[8 * g8 + 4]), b1.x), s5 = fmaf(-2.0f, __uint_as_float(v[8 * g8 + 5]), b1.y);
          const float s6 = fmaf(-2.0f, __uint_as_float(v[8 * g8 + 6]), b1.z), s7 = fmaf(-2.0f, __uint_as_float(v[8 * g8 + 7]), b1.w);
          const float lo = fminf(fminf(fminf(s0, s1), fminf(s2, s3)), fminf(fminf(s4, s5), fminf(s6, s7)));
          flags |= (lo < thr ? 1u : 0u) << (4 * c + g8);
        }
      }
      // Pass 2, ONE copy of the insertion code for the whole kernel: the groups flagged by any lane are read again
      // from TMEM (the accumulator has not been released yet) and their 8 columns pushed in ascending order.
      uint32_t pending = (debug & 16) ? 0u : __reduce_or_sync(kFull, flags);
#pragma unroll 1
      while (pending) {
        const int g = __ffs(pending) - 1;
        pending &= pending - 1;
        uint32_t r[8];
        tmem_ld8(taddr + 8 * g, r);
        const float4 b0 = bn[2 * g], b1 = bn[2 * g + 1];
        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        if ((flags >> g) & 1) {
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float sc = fmaf(-2.0f, __uint_as_float(r[u]), bb[u]);
            if (sc < thr) { top.push(sc, n0 + 8 * g + u + index_offset); thr = top.s[K - 1]; }
          }
        }
      }
      tcgen05_fence_before();
      mbar_arrive(bar_t_empty(acc));
      __syncwarp();
    }
    if (row < qa) {
      const int64_t o = ((int64_t(blockIdx.y) * kEpiParts + half) * qa + row) * K;
#pragma unroll
      for (int k = 0; k < K; ++k) { score[o + k] = top.s[k]; idx[o + k] = top.i[k]; }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// ---- host side ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D float16 row-major (rows, wp) tensor, box = (64 columns, box_rows rows), 128-byte swizzle, zero fill.
static int make_map(CUtensorMap* map, const __half* base, int64_t rows, int wp, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  SF_REQUIRE(fn != nullptr, SF_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  const cuuint64_t dims[2] = {cuuint64_t(wp), cuuint64_t(rows)};
  const cuuint64_t strides[1] = {cuuint64_t(wp) * sizeof(__half)};
  const cuuint32_t box[2] = {cuuint32_t(kBK), cuuint32_t(box_rows)};
  const cuuint32_t elem[2] = {1, 1};
  const CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides, box, elem,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SF_REQUIRE(rc == CUDA_SUCCESS, SF_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", int(rc));
  return SF_OK;
}

template <int K>
static int launch(const CUtensorMap& ma, const CUtensorMap& mb, const float* bnorm, int64_t qa, int64_t qb, int num_kb,
                  int splits, int tiles_per_split, int off, float* score, int32_t* idx, cudaStream_t stream) {
  static bool configured = false;
  if (!configured) {
    SF_CUDA(cudaFuncSetAttribute(topk_tc_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kSmemBytes)));
    configured = true;
  }
  const dim3 grid(unsigned((qa + kBM - 1) / kBM), unsigned(splits));
  static const int debug = getenv("SF_TC_DEBUG") ? atoi(getenv("SF_TC_DEBUG")) : 0;
  topk_tc_kernel<K><<<grid, kThreads, kSmemBytes, stream>>>(ma, mb, bnorm, qa, qb, num_kb, tiles_per_split, off, score, idx,
                                                            debug);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

}  // namespace tc

int launch_topk_tc(const __half* a, int64_t qa, const __half* b, const float* bnorm, int64_t qb, int wp, int k,
                   int index_offset, float* score, int32_t* idx, cudaStream_t stream) {
  using namespace tc;
  SF_REQUIRE(wp % kBK == 0 && wp / kBK <= kMaxKBlocks, SF_ERR_CAPACITY,
             "tensor-core shortlist: padded width %d exceeds %d (use the CUDA-core kernel)", wp, kMaxKBlocks * kBK);
  SF_REQUIRE((reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(b) & 15) == 0, SF_ERR_ARG,
             "tensor-core shortlist: operands must be 16-byte aligned");
  if (qb == 0) {
    SF_CUDA(cudaMemsetAsync(idx, 0xFF, size_t(qa) * k * sizeof(int32_t), stream));
    SF_CUDA(cudaMemsetAsync(score, 0x7F, size_t(qa) * k * sizeof(float), stream));  // NaN-ish sentinel, idx = -1 rules
    return SF_OK;
  }
  CUtensorMap map_a, map_b;
  if (int rc = make_map(&map_a, a, qa, wp, kBM)) return rc;
  if (int rc = make_map(&map_b, b, qb, wp, kBN)) return rc;
  const int m_tiles = int((qa + kBM - 1) / kBM);
  const int n_tiles = int((qb + kBN - 1) / kBN);
  // enough CTAs for ~2 waves of the 148 SMs when the query tiles alone cannot provide them
  int splits = 1;
  if (m_tiles < 2 * 148) splits = std::min(n_tiles, std::max(1, (2 * 148 + m_tiles - 1) / m_tiles));
  const int tiles_per_split = (n_tiles + splits - 1) / splits;
  splits = (n_tiles + tiles_per_split - 1) / tiles_per_split;
  // every CTA emits kEpiParts partial shortlists per row (one per column part of its tiles)
  const int parts = kEpiParts * splits;
  float* part_score = nullptr;
  int32_t* part_idx = nullptr;
  Scratch scratch(stream);
  SF_CUDA(scratch.alloc(&part_score, size_t(parts) * qa * k * sizeof(float)));
  SF_CUDA(scratch.alloc(&part_idx, size_t(parts) * qa * k * sizeof(int32_t)));
  const int num_kb = wp / kBK;
  int rc = SF_OK;
  switch (k) {
    case 1: rc = launch<1>(map_a, map_b, bnorm, qa, qb, num_kb, splits, tiles_per_split, index_offset, part_score, part_idx, stream); break;
    case 2: rc = launch<2>(map_a, map_b, bnorm, qa, qb, num_kb, splits, tiles_per_split, index_offset, part_score, part_idx, stream); break;
    case 4: rc = launch<4>(map_a, map_b, bnorm, qa, qb, num_kb, splits, tiles_per_split, index_offset, part_score, part_idx, stream); break;
    case 8: rc = launch<8>(map_a, map_b, bnorm, qa, qb, num_kb, splits, tiles_per_split, index_offset, part_score, part_idx, stream); break;
    default: rc = launch<16>(map_a, map_b, bnorm, qa, qb, num_kb, splits, tiles_per_split, index_offset, part_score, part_idx, stream); break;
  }
  if (rc != SF_OK) return rc;
  return launch_merge_partials(part_score, part_idx, parts, qa, k, score, idx, stream);
}

}  // namespace sf
