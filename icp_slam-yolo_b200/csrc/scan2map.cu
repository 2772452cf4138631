// scan2map.cu -- scan-to-map ICP against a large map sharded across GPUs (sm_100a).
//
// Same reference loop as the pair kernels (labels_segmentation/icp.py:28-53) with a target set of
// millions of points, for the scan-to-local-map call shape of duc/ICP_LIDAR/mainn.py:297-318.
//
// Round-2 design: EXACT CULLING + EXACT SCAN, two launches per iteration.
//   s2m_prepare_kernel  chunks of 1,024 consecutive map points -> bounding circle (centroid,
//                       radius); s2m_super_kernel: one circle per 32 chunks.  The circle tables
//                       of ALL ranks are replicated on every rank (a few hundred KB), so a rank
//                       can bound a scan point's nearest-neighbour distance over the WHOLE map
//                       without a collective.
//   s2m_search_kernel   one warp per scan point, eight consecutive points per CTA: (1) apply the
//                       pose increment the previous update left pending; (2) upper bound ub of the NN
//                       distance: the distance to the previous iteration's nearest map point (a real
//                       map point), or in the first iteration min over circles of |s - o| + r (two
//                       levels); (2b) the CTA tests the local super-circles once against a ball that
//                       holds the reach circles of its eight points, each warp then only the
//                       survivors; (3) ONE traversal lists every LOCAL chunk whose circle comes within
//                       ub of the point (per-warp list in shared memory); the chunk with the closest
//                       centre is scanned first and tightens the bound, the rest are re-tested and
//                       scanned: exhaustively, behind an exact FP32 filter that skips the points PROVEN
//                       farther than the bound, the survivors in float64 (NumPy's operation order;
//                       exact ties go to the lowest original index, lexicographic warp reduction): the
//                       record it emits is the exact nearest point of this shard among all that can
//                       matter -- no approximate candidate stage, no ambiguity lists, no fallback scan;
//                       (4) the 32-byte record is stored straight into EVERY rank's inbox over
//                       NVLink (peer stores) and the last CTA raises this rank's flag there
//                       (system-scope release): the all-gather is the kernel's epilogue.
//   s2m_update_kernel   waits for the flags of all ranks (system-scope acquire), then per point
//                       the global winner (smaller distance, then lower global index), centred
//                       sums in a fixed order (per-CTA partials, last CTA adds them by CTA index),
//                       closed-form pose, convergence: bit-identical on every rank, so no second
//                       collective is needed.  The increment is applied by the next search.
// A skipped chunk is PROVEN farther from the point than its nearest neighbour, so indices equal
// the float64 brute force (KD-tree) result.  On the benchmark map (16.7 M points along ~100 m of
// wall) a scan point meets ~7 chunks instead of 16,384.
// Replaces: KDTree(B).query(src) (icp.py:37-38), best_fit_transform (icp.py:5-26), the apply /
// convergence steps (icp.py:45-51).
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cub/cub.cuh>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "common.cuh"

namespace {

constexpr int kChunk = 1024;          // map points per bounding circle (512: 2.53 ms, 2048: 2.49 ms against 2.33 ms per alignment)
constexpr int kSuper = 32;            // chunks per second-level circle (one lane each)
constexpr int kSearchWarps = 8;       // warps per CTA of the search kernel
constexpr int kSearchMinCtas = 4;     // 64 registers: 32 resident warps per SM (the kernel is latency-bound:
                                      // 80 registers / 24 warps costs 40 %)
constexpr int kUpdateThreads = 256;
constexpr int kMaxUpdateCtas = 64;
constexpr int kMaxWorld = 32;
constexpr double kUp = 1.000000000001;     // rounds a computed float64 bound outwards
constexpr double kDown = 0.999999999999;
constexpr long long kNoIndex = 0x7fffffffffffffffLL;
constexpr unsigned long long kTimeoutNs = 2000000000ull;    // peer flags: 2 s

struct Circle {           // 32 bytes: one entry of the chunk / super-chunk tables
  double ox, oy, r, pad;  // r < 0: padding entry (no points)
};

// scratch words (uint32) at the start of the caller's scratch buffer; zeroed once by the caller,
// every kernel leaves its ticket at 0
enum { kTicketSearch = 0, kTicketUpdate = 1, kTicketFinish = 2, kScratchHeader = 64 };

__device__ __forceinline__ Circle load_circle(const double* table, int64_t k) {
  const double2 a = __ldg(reinterpret_cast<const double2*>(table) + 2 * k);
  const double2 b = __ldg(reinterpret_cast<const double2*>(table) + 2 * k + 1);
  Circle c;
  c.ox = a.x; c.oy = a.y; c.r = b.x; c.pad = b.y;
  return c;
}

__device__ __forceinline__ double warp_min_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(kFull, v, o));
  return v;
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// peer inbox layout: [2 slots][world][n] records, [2][world] int64 flags, int64 exchange counter
__device__ __forceinline__ b200icp_s2m_record* inbox_records(void* base, int world, int n, int slot, int rank) {
  return reinterpret_cast<b200icp_s2m_record*>(base) + ((int64_t)slot * world + rank) * n;
}
__device__ __forceinline__ long long* inbox_flags(void* base, int world, int n) {
  return reinterpret_cast<long long*>(reinterpret_cast<b200icp_s2m_record*>(base) + (int64_t)2 * world * n);
}

// ------------------------------------------------------------------------------------------
// prepare (optional): Morton order.  Chunks are runs of 1,024 consecutive points, so the culling
// needs an order in which neighbours in memory are neighbours in space.  Accumulated LiDAR scans
// have one; a map that went through a hash-based voxel filter does not.  Sorting the shard once by
// the Morton code of its points (16 bits per axis inside the shard's bounding box) makes the circles
// compact for ANY map.  The scan then runs over the sorted copy; `order[j]` is the original index
// of sorted point j, which is what the records report and what ties are broken on.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long f64_ordered(double v) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double f64_unordered(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// box[0..3] = ordered keys of min x, min y, max x, max y (pre-set to ~0, ~0, 0, 0)
__global__ void __launch_bounds__(256) s2m_bbox_kernel(const void* points, int dtype, int64_t m,
                                                       unsigned long long* box) {
  double x0 = CUDART_INF, y0 = CUDART_INF, x1 = -CUDART_INF, y1 = -CUDART_INF;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += (int64_t)gridDim.x * blockDim.x) {
    const double2 q = load_point(points, dtype, j);
    if (q.x == q.x && q.y == q.y) {
      x0 = fmin(x0, q.x); x1 = fmax(x1, q.x); y0 = fmin(y0, q.y); y1 = fmax(y1, q.y);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    x0 = fmin(x0, __shfl_xor_sync(kFull, x0, o)); x1 = fmax(x1, __shfl_xor_sync(kFull, x1, o));
    y0 = fmin(y0, __shfl_xor_sync(kFull, y0, o)); y1 = fmax(y1, __shfl_xor_sync(kFull, y1, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(box + 0, f64_ordered(x0)); atomicMin(box + 1, f64_ordered(y0));
    atomicMax(box + 2, f64_ordered(x1)); atomicMax(box + 3, f64_ordered(y1));
  }
}

__device__ __forceinline__ unsigned spread16(unsigned v) {      // abcd -> 0a0b0c0d
  v = (v | (v << 8)) & 0x00ff00ffu;
  v = (v | (v << 4)) & 0x0f0f0f0fu;
  v = (v | (v << 2)) & 0x33333333u;
  v = (v | (v << 1)) & 0x55555555u;
  return v;
}

__global__ void __launch_bounds__(256) s2m_morton_kernel(const void* points, int dtype, int64_t m,
                                                         const unsigned long long* __restrict__ box,
                                                         unsigned* __restrict__ keys, int32_t* __restrict__ idx) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const double x0 = f64_unordered(box[0]), y0 = f64_unordered(box[1]);
  const double ext = fmax(fmax(f64_unordered(box[2]) - x0, f64_unordered(box[3]) - y0), 1e-300);
  const double2 q = load_point(points, dtype, j);
  const double fx = (q.x - x0) / ext * 65535.0, fy = (q.y - y0) / ext * 65535.0;   // one scale: square cells
  const unsigned qx = (unsigned)fmin(fmax(fx, 0.0), 65535.0), qy = (unsigned)fmin(fmax(fy, 0.0), 65535.0);
  keys[j] = spread16(qx) | (spread16(qy) << 1);
  idx[j] = (int32_t)j;
}

__global__ void __launch_bounds__(256) s2m_gather_kernel(const void* points, int dtype, int64_t m,
                                                         const int32_t* __restrict__ order, void* sorted) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  if (dtype == B200ICP_F64) reinterpret_cast<double2*>(sorted)[j] = reinterpret_cast<const double2*>(points)[order[j]];
  else reinterpret_cast<float2*>(sorted)[j] = reinterpret_cast<const float2*>(points)[order[j]];
}

struct SortWs {
  int64_t box, keys_in, keys_out, idx_in, cub, total;
  size_t cub_bytes;
};

SortWs sort_layout(int64_t m) {
  auto up = [](int64_t b) { return (b + 255) / 256 * 256; };
  SortWs w;
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const unsigned*)nullptr, (unsigned*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, (int)m);
  w.cub_bytes = cub_bytes;
  int64_t off = 0;
  w.box = off;      off += 256;
  w.keys_in = off;  off += up(m * 4);
  w.keys_out = off; off += up(m * 4);
  w.idx_in = off;   off += up(m * 4);
  w.cub = off;      off += up((int64_t)cub_bytes);
  w.total = off;
  return w;
}

// ------------------------------------------------------------------------------------------
// prepare: bounding circle of every chunk, then of every 32 chunks
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) s2m_prepare_kernel(const void* points, int dtype, int64_t m,
                                                          int n_chunks, double* chunk_circle) {
  __shared__ double sred[8][2];
  __shared__ double rred[8];
  const int c = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (c >= n_chunks) {                                 // padding entry of the last super-chunk
    if (tid == 0) { chunk_circle[4 * c] = 0.0; chunk_circle[4 * c + 1] = 0.0; chunk_circle[4 * c + 2] = -1.0; chunk_circle[4 * c + 3] = 0.0; }
    return;
  }
  const int64_t j0 = (int64_t)c * kChunk;
  const int cnt = (int)min((int64_t)kChunk, m - j0);
  double sx = 0.0, sy = 0.0;
  for (int j = tid; j < cnt; j += blockDim.x) {
    const double2 q = load_point(points, dtype, j0 + j);
    sx += q.x; sy += q.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sx += __shfl_xor_sync(kFull, sx, o);
    sy += __shfl_xor_sync(kFull, sy, o);
  }
  if (lane == 0) { sred[warp][0] = sx; sred[warp][1] = sy; }
  __syncthreads();
  double tx = 0.0, ty = 0.0;
  for (int w = 0; w < 8; ++w) { tx += sred[w][0]; ty += sred[w][1]; }
  const double ox = tx / (double)cnt, oy = ty / (double)cnt;
  double r2 = 0.0;
  for (int j = tid; j < cnt; j += blockDim.x) {
    const double2 q = load_point(points, dtype, j0 + j);
    const double dx = q.x - ox, dy = q.y - oy;
    r2 = fmax(r2, dx * dx + dy * dy);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) r2 = fmax(r2, __shfl_xor_sync(kFull, r2, o));
  if (lane == 0) rred[warp] = r2;
  __syncthreads();
  if (tid == 0) {
    double r = 0.0;
    for (int w = 0; w < 8; ++w) r = fmax(r, rred[w]);
    chunk_circle[4 * c] = ox; chunk_circle[4 * c + 1] = oy;
    chunk_circle[4 * c + 2] = sqrt(r) * kUp + 1e-300;          // >= the true radius
    chunk_circle[4 * c + 3] = 0.0;
  }
}

__global__ void __launch_bounds__(32) s2m_super_kernel(const double* __restrict__ chunk_circle,
                                                       double* __restrict__ super_circle) {
  const int s = blockIdx.x, lane = threadIdx.x;
  const Circle c = load_circle(chunk_circle, (int64_t)s * kSuper + lane);
  const bool valid = c.r >= 0.0;
  double sx = valid ? c.ox : 0.0, sy = valid ? c.oy : 0.0, cnt = valid ? 1.0 : 0.0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sx += __shfl_xor_sync(kFull, sx, o);
    sy += __shfl_xor_sync(kFull, sy, o);
    cnt += __shfl_xor_sync(kFull, cnt, o);
  }
  double ox = 0.0, oy = 0.0, r = -1.0;
  if (cnt > 0.0) {
    ox = sx / cnt; oy = sy / cnt;
    double rr = 0.0;
    if (valid) {
      const double dx = c.ox - ox, dy = c.oy - oy;
      rr = sqrt(dx * dx + dy * dy) * kUp + c.r;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rr = fmax(rr, __shfl_xor_sync(kFull, rr, o));
    r = rr * kUp;
  }
  if (lane == 0) {
    super_circle[4 * s] = ox; super_circle[4 * s + 1] = oy; super_circle[4 * s + 2] = r; super_circle[4 * s + 3] = 0.0;
  }
}

// ------------------------------------------------------------------------------------------
// init
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) s2m_init_kernel(const void* scan, int dtype, int n,
                                                       const double* init_pose, double* src64,
                                                       double* prev_nn, b200icp_s2m_state* state) {
  double R00 = 1, R01 = 0, R10 = 0, R11 = 1, T0 = 0, T1 = 0;
  if (init_pose) { R00 = init_pose[0]; R01 = init_pose[1]; R10 = init_pose[2]; R11 = init_pose[3]; T0 = init_pose[4]; T1 = init_pose[5]; }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double2 q = load_point(scan, dtype, i);
    src64[2 * i] = init_pose ? R00 * q.x + R01 * q.y + T0 : q.x;
    src64[2 * i + 1] = init_pose ? R10 * q.x + R11 * q.y + T1 : q.y;
    if (prev_nn) { prev_nn[2 * i] = CUDART_NAN; prev_nn[2 * i + 1] = CUDART_NAN; }   // "no previous neighbour"
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    state->pose_total[0] = R00; state->pose_total[1] = R01; state->pose_total[2] = R10;
    state->pose_total[3] = R11; state->pose_total[4] = T0; state->pose_total[5] = T1;
    state->pose_last[0] = 1; state->pose_last[1] = 0; state->pose_last[2] = 0;
    state->pose_last[3] = 1; state->pose_last[4] = 0; state->pose_last[5] = 0;
    state->error = CUDART_INF; state->mean_d2 = CUDART_INF; state->prev_error = 0.0;   // icp.py:33
    state->iterations = 0; state->inliers = 0; state->done = (n <= 0) ? 1 : 0; state->applied = 0;
  }
}

// src <- R_last src + t_last for the increment an update left pending (icp.py:45)
__device__ __forceinline__ double2 apply_pending(const b200icp_s2m_state* st, double2 s) {
  const double cs = st->pose_last[0], sn = st->pose_last[2], tx = st->pose_last[4], ty = st->pose_last[5];
  return make_double2(cs * s.x - sn * s.y + tx, sn * s.x + cs * s.y + ty);
}

// ------------------------------------------------------------------------------------------
// search: one warp per scan point (see the header of this file)
// ------------------------------------------------------------------------------------------
struct SearchArgs {
  const void* points;          // this rank's shard as it is scanned (the Morton-sorted copy if there is one)
  const int32_t* order;        // sorted position -> original local index, or NULL (scanned in the given order)
  int64_t m, global_offset;
  int dtype;
  const double* chunk_circle;  // circles of the whole map (all ranks, rank order)
  const double* super_circle;
  int n_chunks_total;          // multiple of 32
  int first_local_chunk;       // multiple of 32
  int n_local_chunks;          // padded, multiple of 32
  double* src64;
  const double* prev_nn;       // [n][2] nearest map point of the previous iteration (NaN: none)
  int n;
  b200icp_s2m_record* records; // local output [n] (NULL when peers are used)
  void* const* peers;          // device array of `world` inbox addresses, or NULL
  int world, rank;
  b200icp_s2m_state* state;
  unsigned* scratch;
};

// Is the circle within `reach` of the point?  (squared, rounded so that a true hit is never lost)
__device__ __forceinline__ bool circle_hit(const Circle& c, double sx, double sy, double ub) {
  if (!(c.r >= 0.0)) return false;
  const double dx = sx - c.ox, dy = sy - c.oy, reach = ub + c.r;
  return (dx * dx + dy * dy) * kDown <= reach * reach;
}

// Exhaustive float64 scan of one chunk for one point: lanes stride over the chunk, eight
// independent loads in flight per lane.
// (bd, bp): best squared distance and its position in the scanned array.  On exact ties the lowest
// ORIGINAL index wins whatever the order the chunks are scanned in (the closest chunk goes first):
// the position itself when the map is scanned in its given order, order[] in a Morton-sorted copy.
__device__ __forceinline__ void consider(const SearchArgs& a, double d, long long pos, double& bd, long long& bp) {
  if (d <= bd) {
    if (d < bd) { bd = d; bp = pos; }
    else if (bp != kNoIndex && (a.order ? a.order[pos] < a.order[bp] : pos < bp)) bp = pos;   // exact tie
  }
}

// FP32 filter in front of the exact float64 test (float32 maps).  A map point can only change the
// result if its exact distance is <= the best so far.  With s32 = RN(s) and the float32 point q
// (exact), the FP32 value d32 = RN(dx^2 + dy^2), dx = RN(q.x - s32.x), carries a relative error
// < 2^-21 in the distance plus the absolute error of rounding s: |s - s32| <= 2^-24 (|s.x| + |s.y|)
// per axis.  So  dist >= sqrt(d32) (1 - 2^-21) - A,  A = 5e-7 (|s.x| + |s.y|) + 1e-20  (more than 4 x
// the rounding of s), and every point with  d32 > thr = RU(((sqrt(best) + A) * 1.000004)^2)  is PROVEN
// farther than the best: it is skipped without the two conversions and five float64 operations of
// the exact test.  Points that pass go through `consider` unchanged, so the result is bit for bit the
// one of the unfiltered scan.  `best` may be the best of the WHOLE warp (another lane's point at
// exactly that distance still passes: d <= best).
struct Fp32Filter {
  float sx, sy;      // RN(s)
  float thr;         // skip threshold on d32 (+inf: no bound yet)
  double slack;      // A
};

__device__ __forceinline__ float filter_threshold(double best, double slack) {
  if (!(best < CUDART_INF)) return CUDART_INF_F;
  const double r = (sqrt(best) + slack) * 1.000004;
  return __double2float_ru(r * r);
}

// Eight points of one lane (positions pos0 + 32 u) against the point (sx, sy).
__device__ __forceinline__ void scan_round(const SearchArgs& a, const float2 (&q)[8], int64_t pos0, double sx,
                                           double sy, double& bd, long long& bp, Fp32Filter& f) {
  float d32[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const float dx = q[u].x - f.sx, dy = q[u].y - f.sy;
    d32[u] = fmaf(dx, dx, dy * dy);
  }
  const float lo = fminf(fminf(fminf(d32[0], d32[1]), fminf(d32[2], d32[3])),
                         fminf(fminf(d32[4], d32[5]), fminf(d32[6], d32[7])));
  if (lo <= f.thr) {                          // rare: the filter starts from the bound of the NN distance
    const double before = bd;
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (d32[u] <= f.thr)
        consider(a, dist2_f64(sx, sy, make_double2((double)q[u].x, (double)q[u].y)), pos0 + 32 * u, bd, bp);
    if (bd < before) f.thr = fminf(f.thr, filter_threshold(bd, f.slack));
  }
}

__device__ __forceinline__ void scan_chunk(const SearchArgs& a, int lc, double sx, double sy, int lane,
                                           double& bd, long long& bp, Fp32Filter& f) {
  const int64_t j0 = (int64_t)lc * kChunk;
  const int cnt = (int)min((int64_t)kChunk, a.m - j0);
  int j = lane;
  if (a.dtype == B200ICP_F32) {
    const float2* __restrict__ p = reinterpret_cast<const float2*>(a.points) + j0;
    for (; j + 224 < cnt; j += 256) {
      float2 q[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) q[u] = __ldg(p + j + 32 * u);
      scan_round(a, q, j0 + j, sx, sy, bd, bp, f);
    }
  } else {
    const double2* __restrict__ p = reinterpret_cast<const double2*>(a.points) + j0;
    for (; j + 96 < cnt; j += 128) {
      double2 q[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) q[u] = __ldg(p + j + 32 * u);
#pragma unroll
      for (int u = 0; u < 4; ++u) consider(a, dist2_f64(sx, sy, q[u]), j0 + j + 32 * u, bd, bp);
    }
  }
  for (; j < cnt; j += 32) consider(a, dist2_f64(sx, sy, load_point(a.points, a.dtype, j0 + j)), j0 + j, bd, bp);
}

constexpr int kSuperBlock = 1024;     // super-chunks per traversal block: one candidate bit per lane and trip
constexpr int kListCap = 64;          // listed candidate chunks per scan point (more: second traversal)
constexpr int kSupCap = 64;           // super-chunks the CTA's ball may meet (more: per-warp traversal of all)
#ifndef S2M_TIMING
#define S2M_TIMING 0
#endif
#if S2M_TIMING
__device__ unsigned long long g_s2m_clk[8];   // debug builds only: per-phase cycles summed over warps
#define S2M_TICK(slot)                                                          \
  do {                                                                          \
    const long long now_ = clock64();                                           \
    if (lane == 0) atomicAdd(&g_s2m_clk[slot], (unsigned long long)(now_ - tick_)); \
    tick_ = now_;                                                               \
  } while (0)
#else
#define S2M_TICK(slot) do { } while (0)
#endif

__global__ void __launch_bounds__(kSearchWarps * 32, kSearchMinCtas) s2m_search_kernel(const SearchArgs a) {
  __shared__ __align__(16) b200icp_s2m_record srec[kSearchWarps];     // the CTA's records, staged for the peer stores
  __shared__ int clist[kSearchWarps][kListCap];                       // per warp: the chunks within reach of its point
  __shared__ double2 cta_pt[kSearchWarps];                            // the CTA's points and bounds
  __shared__ double cta_ub[kSearchWarps];
  __shared__ int sup_list[kSupCap];                                   // local super-chunks within reach of the CTA
  __shared__ int sup_count;
  b200icp_s2m_state* st = a.state;
  if (st->done) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // One warp per scan point.  (Several warps per point, each scanning every k-th listed chunk, were
  // measured: the repeated circle traversal costs more than the shorter load chain saves --
  // profiles/r2_kernel_tuning.md.)
  const int i = blockIdx.x * kSearchWarps + warp;
  const bool active = i < a.n;
  const bool pending = st->applied < st->iterations;
  long long seq = 0;
  int slot = 0;
  if (a.peers) {
    seq = *(inbox_flags(a.peers[a.rank], a.world, a.n) + 2 * a.world) + 1;   // exchange counter of this rank
    slot = (int)(seq & 1);
  }
#if S2M_TIMING
  long long tick_ = clock64();
#endif
  double bd = CUDART_INF;
  long long bj = kNoIndex;
  double2 s = make_double2(0.0, 0.0);
  double ub = 0.0, cd = CUDART_INF, cr = 0.0;   // bound of the NN distance; closest chunk centre among the candidates
  int cc = -1, count = 0;
  Fp32Filter flt;
  flt.sx = 0.f; flt.sy = 0.f; flt.thr = CUDART_INF_F; flt.slack = 0.0;
  int* const mylist = clist[warp];
  const int first_super = a.first_local_chunk / kSuper, local_supers = a.n_local_chunks / kSuper;
  if (active) {
    s = make_double2(a.src64[2 * i], a.src64[2 * i + 1]);
    if (pending) {
      s = apply_pending(st, s);
      if (lane == 0) { a.src64[2 * i] = s.x; a.src64[2 * i + 1] = s.y; }
    }
    // ---- (2) upper bound of the nearest-neighbour distance over the whole map
    const double px = a.prev_nn ? a.prev_nn[2 * i] : CUDART_NAN, py = a.prev_nn ? a.prev_nn[2 * i + 1] : CUDART_NAN;
    if (px == px) {
      ub = sqrt(dist2_f64(s.x, s.y, make_double2(px, py)) * kUp) * kUp;
    } else {
      const int n_super = a.n_chunks_total / kSuper;
      double ub0 = CUDART_INF;
      for (int k = lane; k < n_super; k += 32) {
        const Circle c = load_circle(a.super_circle, k);
        if (c.r >= 0.0) {
          const double dx = s.x - c.ox, dy = s.y - c.oy;
          ub0 = fmin(ub0, sqrt(dx * dx + dy * dy) * kUp + c.r);
        }
      }
      ub0 = warp_min_f64(ub0);
      double ub1 = ub0;
      for (int k0 = 0; k0 < n_super; k0 += 32) {
        const bool near = k0 + lane < n_super && circle_hit(load_circle(a.super_circle, k0 + lane), s.x, s.y, ub0);
        unsigned mask = __ballot_sync(kFull, near);
        while (mask) {
          const int k = k0 + __ffs(mask) - 1;
          mask &= mask - 1;
          const Circle c = load_circle(a.chunk_circle, (int64_t)k * kSuper + lane);
          if (c.r >= 0.0) {
            const double dx = s.x - c.ox, dy = s.y - c.oy;
            ub1 = fmin(ub1, sqrt(dx * dx + dy * dy) * kUp + c.r);
          }
        }
      }
      ub = warp_min_f64(ub1) * kUp;
    }
  }
  // ---- (2b) the eight points of a CTA are neighbours on the scan, so their reach circles nearly
  // coincide: the CTA tests the local super-circles ONCE against a ball that contains all eight
  // (centre = the first point, radius = max_w(|s_w - s_0| + ub_w)) -- 256 threads, one or two
  // circles each -- and every warp then tests only the few survivors with its own (s, ub).  A
  // super-circle within reach of point w is within reach of the ball (triangle inequality), so the
  // per-warp hit sets are unchanged.  More survivors than the list holds (first iteration): every
  // warp walks all super-circles itself as before.
  int nsup = -1;                               // -1: no CTA list
  {
    if (lane == 0) {
      cta_pt[warp] = make_double2(s.x, s.y);
      cta_ub[warp] = active ? ub : -1.0;
    }
    if (threadIdx.x == 0) sup_count = 0;
    __syncthreads();
    const double2 c0 = cta_pt[0];              // warp 0 of a launched CTA always has a point
    double R = 0.0;
#pragma unroll
    for (int w = 0; w < kSearchWarps; ++w) {
      const double ubw = cta_ub[w];
      if (ubw >= 0.0) {
        const double dx = cta_pt[w].x - c0.x, dy = cta_pt[w].y - c0.y;
        R = fmax(R, sqrt(dx * dx + dy * dy) * kUp + ubw);
      }
    }
    R *= kUp;
    for (int k = threadIdx.x; k < local_supers; k += kSearchWarps * 32) {
      if (circle_hit(load_circle(a.super_circle, first_super + k), c0.x, c0.y, R)) {
        const int at = atomicAdd(&sup_count, 1);
        if (at < kSupCap) sup_list[at] = k;
      }
    }
    __syncthreads();
    nsup = sup_count <= kSupCap ? sup_count : -1;
  }
  if (active) {
    // ---- (3) exact float64 scan of every local chunk within reach.  ONE traversal of the local
    // circles lists the chunks within the bound (ascending, per-warp list in shared memory) and
    // finds the one whose centre is closest.  That chunk is scanned first; if the bound was wider
    // than it (the scan moved a lot, or this is the first iteration) its best distance becomes the
    // bound and the listed chunks are re-tested against it -- the same predicate on a superset, so
    // the set of scanned chunks is exactly the one a second traversal would find.  A list that
    // overflows (first iterations: hundreds of chunks within a loose bound) falls back to that
    // second traversal.
    S2M_TICK(0);                               // point, pending increment, bound
    flt.sx = (float)s.x; flt.sy = (float)s.y;
    flt.slack = 5e-7 * (fabs(s.x) + fabs(s.y)) + 1e-20;        // + underflow of the FP32 squares
    // a real map point lies within ub of s (the previous nearest neighbour, or a point of the circle
    // that gave the bound), possibly in another shard: nothing farther than ub can be the global
    // nearest neighbour, so the filter starts from ub instead of +inf
    flt.thr = filter_threshold(ub * ub * kUp, flt.slack);
    // chunk level: the 32 chunk circles of every hit super-chunk, one per lane; the circles of the
    // next hit super-chunk are loaded while the current ones are tested
    auto visit = [&](unsigned smask, auto super_of) {
      int ks = -1;
      Circle c;
      c.ox = 0.0; c.oy = 0.0; c.r = -1.0; c.pad = 0.0;
      if (smask) {
        ks = super_of(__ffs(smask) - 1);                               // local super-chunk
        smask &= smask - 1;
        c = load_circle(a.chunk_circle, (int64_t)(first_super + ks) * kSuper + lane);
      }
      while (ks >= 0) {
        int kn = -1;
        Circle cn = c;
        if (smask) {
          kn = super_of(__ffs(smask) - 1);
          smask &= smask - 1;
          cn = load_circle(a.chunk_circle, (int64_t)(first_super + kn) * kSuper + lane);
        }
        const bool hit = circle_hit(c, s.x, s.y, ub);
        if (hit) {
          const double dx = s.x - c.ox, dy = s.y - c.oy, d = dx * dx + dy * dy;
          if (d < cd) { cd = d; cr = c.r; cc = ks * kSuper + lane; }
        }
        const unsigned cmask = __ballot_sync(kFull, hit);
        const int at = count + __popc(cmask & ((1u << lane) - 1u));
        if (hit && at < kListCap) mylist[at] = ks * kSuper + lane;
        count += __popc(cmask);
        ks = kn;
        c = cn;
      }
    };
    if (nsup >= 0) {                           // the CTA's survivors (any order: ties are decided on positions)
      for (int q0 = 0; q0 < nsup; q0 += 32) {
        const int k = q0 + lane < nsup ? sup_list[q0 + lane] : -1;
        const bool near = k >= 0 && circle_hit(load_circle(a.super_circle, first_super + k), s.x, s.y, ub);
        visit(__ballot_sync(kFull, near), [&](int bit) { return sup_list[q0 + bit]; });
      }
    } else {
      for (int b0 = 0; b0 < local_supers; b0 += kSuperBlock) {
        const int trips = (min(kSuperBlock, local_supers - b0) + 31) >> 5;
        unsigned my = 0;                      // bit t: super b0 + 32 t + lane is within reach (loads independent)
        for (int t = 0; t < trips; ++t) {
          const int k = b0 + 32 * t + lane;
          const bool near = k < local_supers && circle_hit(load_circle(a.super_circle, first_super + k), s.x, s.y, ub);
          my |= (near ? 1u : 0u) << t;
        }
        if (!__any_sync(kFull, my != 0)) continue;
        for (int t = 0; t < trips; ++t)
          visit(__ballot_sync(kFull, (my >> t) & 1u), [&](int bit) { return b0 + 32 * t + bit; });
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(kFull, cd, o), orr = __shfl_xor_sync(kFull, cr, o);
      const int oc = __shfl_xor_sync(kFull, cc, o);
      if (od < cd || (od == cd && oc >= 0 && (cc < 0 || oc < cc))) { cd = od; cr = orr; cc = oc; }
    }
    __syncwarp();                              // the list is read by every lane
    S2M_TICK(1);                               // traversal
  }
  if (active) {
    if (count <= kListCap) {
      bool tightened = false;
      if (cc >= 0 && count > 1) {              // closest chunk first; its result is kept
        scan_chunk(a, cc, s.x, s.y, lane, bd, bj, flt);
        const double wbest = warp_min_f64(bd);                 // the warp's best: every lane filters on it
        flt.thr = fminf(flt.thr, filter_threshold(wbest, flt.slack));
        if (ub > cr) {
          const double t2 = fmin(ub, sqrt(wbest * kUp) * kUp);
          tightened = t2 < ub;
          ub = t2;
        }
      } else {
        cc = -1;
      }
      for (int e = 0; e < count; ++e) {
        const int lc = mylist[e];
        if (lc == cc) continue;
        if (tightened &&
            !circle_hit(load_circle(a.chunk_circle, (int64_t)first_super * kSuper + lc), s.x, s.y, ub)) continue;
        scan_chunk(a, lc, s.x, s.y, lane, bd, bj, flt);
      }
    } else {
      if (cc >= 0 && ub > cr) {               // the bound is wider than the closest chunk: tighten it there
        double td = CUDART_INF;
        long long tj = kNoIndex;
        Fp32Filter tf = flt;
        scan_chunk(a, cc, s.x, s.y, lane, td, tj, tf);
        td = warp_min_f64(td);
        flt.thr = fminf(flt.thr, filter_threshold(td, flt.slack));   // a real map point at distance td exists
        ub = fmin(ub, sqrt(td * kUp) * kUp);
      }
      for (int b0 = 0; b0 < local_supers; b0 += kSuperBlock) {
        const int trips = (min(kSuperBlock, local_supers - b0) + 31) >> 5;
        unsigned my = 0;
        for (int t = 0; t < trips; ++t) {
          const int k = b0 + 32 * t + lane;
          const bool near = k < local_supers && circle_hit(load_circle(a.super_circle, first_super + k), s.x, s.y, ub);
          my |= (near ? 1u : 0u) << t;
        }
        if (!__any_sync(kFull, my != 0)) continue;
        for (int t = 0; t < trips; ++t) {
          unsigned smask = __ballot_sync(kFull, (my >> t) & 1u);
          while (smask) {
            const int ks = b0 + 32 * t + __ffs(smask) - 1;
            smask &= smask - 1;
            const Circle c = load_circle(a.chunk_circle, (int64_t)(first_super + ks) * kSuper + lane);
            unsigned cmask = __ballot_sync(kFull, circle_hit(c, s.x, s.y, ub));
            while (cmask) {
              const int lc = ks * kSuper + __ffs(cmask) - 1;           // local chunk, ascending
              cmask &= cmask - 1;
              scan_chunk(a, lc, s.x, s.y, lane, bd, bj, flt);
            }
          }
        }
      }
    }
  }
  S2M_TICK(2);                                 // scans
  if (active) {
    long long bo = (bj != kNoIndex && a.order) ? (long long)a.order[bj] : bj;   // original local index
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {                       // lexicographic (distance, original index)
      const double od = __shfl_xor_sync(kFull, bd, o);
      const long long oo = __shfl_xor_sync(kFull, bo, o), oj = __shfl_xor_sync(kFull, bj, o);
      if (od < bd || (od == bd && oo < bo)) { bd = od; bo = oo; bj = oj; }
    }
    b200icp_s2m_record rec;
    rec.d2 = bd; rec.gidx = kNoIndex; rec.bx = 0.0; rec.by = 0.0;        // "none": the NN is in another shard
    if (bj != kNoIndex) {
      const double2 b = load_point(a.points, a.dtype, bj);
      rec.gidx = a.global_offset + bo; rec.bx = b.x; rec.by = b.y;
    }
    if (lane == 0) {
      if (a.peers) srec[warp] = rec;
      else a.records[i] = rec;
    }
  }
  // ---- (4) all-gather as peer stores: the CTA's records are contiguous in every inbox, so warp w
  // sends them to rank w, w + 8, ... as ONE coalesced store of up to 256 bytes (lane l: 8 bytes)
  // instead of eight 32-byte stores per point -- NVLink moves few large packets much faster than
  // many small ones (profiles/r2_kernel_tuning.md)
  if (a.peers) {
    __syncthreads();
    const int first = blockIdx.x * kSearchWarps;
    const int words = min(kSearchWarps, a.n - first) * 4;               // 8-byte words to send
    for (int r = warp; r < a.world; r += kSearchWarps) {
      double* dst = reinterpret_cast<double*>(inbox_records(a.peers[r], a.world, a.n, slot, a.rank) + first);
      if (lane < words) dst[lane] = reinterpret_cast<const double*>(srec)[lane];
    }
  }
  S2M_TICK(3);                                 // record, peer stores
  // last CTA: the pending increment is applied everywhere; raise this rank's flag on every rank.
  // One system-scope fence per CTA (after the barrier: cumulative over the stores of all its warps)
  // orders the records before the ticket, the ticket chain before the last CTA's fence and flag.
  __syncthreads();
  S2M_TICK(4);                                 // wait for the CTA's slowest warp
  if (threadIdx.x == 0) {
    if (a.peers) __threadfence_system(); else __threadfence();
    const unsigned ticket = atomicAdd(a.scratch + kTicketSearch, 1u);
    if (ticket == gridDim.x - 1) {
      a.scratch[kTicketSearch] = 0u;
      if (pending) st->applied = st->iterations;
      if (a.peers) {
        __threadfence_system();
        for (int r = 0; r < a.world; ++r) {
          long long* flag = inbox_flags(a.peers[r], a.world, a.n) + slot * a.world + a.rank;
          asm volatile("st.release.sys.global.s64 [%0], %1;" ::"l"(flag), "l"(seq) : "memory");
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// update: global winner per point, centred sums in a fixed order, pose, convergence.  Every rank
// runs it on the same records and reaches bit-identical state.
// ------------------------------------------------------------------------------------------
struct UpdateArgs {
  const b200icp_s2m_record* records_all;   // [n_ranks][n], or NULL when `inbox` is used
  void* inbox;                             // this rank's peer inbox, or NULL
  int n_ranks;
  const double* src64;
  double* prev_nn;
  int n;
  int max_iterations;
  double tolerance, max_corr_dist;
  int32_t* idx_out;
  b200icp_s2m_state* state;
  unsigned* scratch;
};

__global__ void __launch_bounds__(kUpdateThreads) s2m_update_kernel(const UpdateArgs a) {
  __shared__ double red[kUpdateThreads / 32][12];
  __shared__ double tot[12];
  __shared__ int timed_out;
  b200icp_s2m_state* st = a.state;
  if (st->done) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool pending = st->applied < st->iterations;       // only when no search ran in between (not in run())
  const b200icp_s2m_record* recs = a.records_all;
  long long seq = 0;
  if (a.inbox) {                                           // wait for the records of every rank
    long long* flags = inbox_flags(a.inbox, a.n_ranks, a.n);
    seq = flags[2 * a.n_ranks] + 1;
    const int slot = (int)(seq & 1);
    if (tid == 0) timed_out = 0;
    __syncthreads();
    if (tid < a.n_ranks) {
      const long long* f = flags + slot * a.n_ranks + tid;
      const unsigned long long t0 = global_timer_ns();
      long long v = 0;
      while (true) {
        asm volatile("ld.acquire.sys.global.s64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
        if (v >= seq) break;
        if (global_timer_ns() - t0 > kTimeoutNs) { timed_out = 1; break; }   // a peer is gone: fail, do not hang
      }
    }
    __syncthreads();
    if (timed_out) {
      if (tid == 0) st->done = 2;
      return;
    }
    recs = inbox_records(a.inbox, a.n_ranks, a.n, slot, 0);
  }
  const bool use_gate = a.max_corr_dist > 0.0 && isfinite(a.max_corr_dist);
  double2 o = make_double2(a.src64[0], a.src64[1]);        // any common origin keeps the sums small
  if (pending) o = apply_pending(st, o);
  double r[11] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = blockIdx.x * kUpdateThreads + tid; i < a.n; i += gridDim.x * kUpdateThreads) {
    const double4* p = reinterpret_cast<const double4*>(recs + i);
    double4 w = *p;                                          // d2, gidx (bits), bx, by
    for (int g = 1; g < a.n_ranks; ++g) {
      const double4 c = *reinterpret_cast<const double4*>(recs + (int64_t)g * a.n + i);
      const long long cj = __double_as_longlong(c.y), wj = __double_as_longlong(w.y);
      if (c.x < w.x || (c.x == w.x && cj < wj)) w = c;
    }
    if (a.idx_out) a.idx_out[i] = (int32_t)__double_as_longlong(w.y);
    a.prev_nn[2 * i] = w.z; a.prev_nn[2 * i + 1] = w.w;
    const double dist = sqrt(w.x);
    if (!use_gate || dist < a.max_corr_dist) {
      double2 s = make_double2(a.src64[2 * i], a.src64[2 * i + 1]);
      if (pending) s = apply_pending(st, s);
      const double ax = s.x - o.x, ay = s.y - o.y;
      const double qx = w.z - o.x, qy = w.w - o.y;
      r[0] += ax; r[1] += ay; r[2] += qx; r[3] += qy;
      r[4] = fma(ax, qx, r[4]); r[5] = fma(ax, qy, r[5]);
      r[6] = fma(ay, qx, r[6]); r[7] = fma(ay, qy, r[7]);
      r[8] += dist; r[9] += w.x; r[10] += 1.0;
    }
  }
#pragma unroll
  for (int q = 0; q < 11; ++q) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) r[q] += __shfl_xor_sync(kFull, r[q], s);
  }
  if (lane == 0) {
#pragma unroll
    for (int q = 0; q < 11; ++q) red[warp][q] = r[q];
  }
  __syncthreads();
  double* partials = reinterpret_cast<double*>(a.scratch + kScratchHeader);      // [ctas][12]
  if (tid < 11) {
    double acc = 0.0;
    for (int w = 0; w < kUpdateThreads / 32; ++w) acc += red[w][tid];
    partials[blockIdx.x * 12 + tid] = acc;
    __threadfence();
  }
  __syncthreads();
  __shared__ unsigned ticket;
  if (tid == 0) ticket = atomicAdd(a.scratch + kTicketUpdate, 1u);
  __syncthreads();
  if (ticket != gridDim.x - 1) return;
  // ---- last CTA: add the partials by CTA index (fixed order), solve, decide
  // (all partials are fetched at once by the whole CTA -- one memory round trip instead of one per
  // CTA -- and then added in CTA order from shared memory: the same additions, the same bits)
  __threadfence();
  __shared__ double part[kMaxUpdateCtas * 12];
  for (unsigned q = tid; q < gridDim.x * 12u; q += kUpdateThreads) part[q] = __ldcg(partials + q);
  __syncthreads();
  if (tid < 11) {
    double acc = 0.0;
    for (unsigned c = 0; c < gridDim.x; ++c) acc += part[c * 12 + tid];
    tot[tid] = acc;
  }
  __syncthreads();
  if (tid != 0) return;
  a.scratch[kTicketUpdate] = 0u;
  if (a.inbox) inbox_flags(a.inbox, a.n_ranks, a.n)[2 * a.n_ranks] = seq;      // this exchange is consumed
  const double cnt = tot[10];
  if (cnt < 0.5) {               // every correspondence gated out: stop, search not counted
    st->error = CUDART_INF; st->mean_d2 = CUDART_INF; st->inliers = 0; st->done = 1;
    return;
  }
  const double inv = 1.0 / cnt;
  const double max_ = tot[0] * inv, may_ = tot[1] * inv, mbx = tot[2] * inv, mby = tot[3] * inv;
  const double mean_error = tot[8] * inv;                          // icp.py:48
  const double h00 = fma(-tot[0], mbx, tot[4]), h01 = fma(-tot[0], mby, tot[5]);
  const double h10 = fma(-tot[1], mbx, tot[6]), h11 = fma(-tot[1], mby, tot[7]);
  const double num = h01 - h10, den = h00 + h11;
  const double h2 = fma(num, num, den * den);
  double cs = 1.0, sn = 0.0;
  if (h2 > 0.0) { const double rh = rsqrt(h2); cs = den * rh; sn = num * rh; }
  const double cax = o.x + max_, cay = o.y + may_;
  const double tx = (o.x + mbx) - (cs * cax - sn * cay);            // icp.py:25
  const double ty = (o.y + mby) - (sn * cax + cs * cay);
  const double R00 = st->pose_total[0], R01 = st->pose_total[1];
  const double R10 = st->pose_total[2], R11 = st->pose_total[3];
  const double T0 = st->pose_total[4], T1 = st->pose_total[5];
  st->pose_total[0] = cs * R00 - sn * R10; st->pose_total[1] = cs * R01 - sn * R11;
  st->pose_total[2] = sn * R00 + cs * R10; st->pose_total[3] = sn * R01 + cs * R11;
  st->pose_total[4] = cs * T0 - sn * T1 + tx; st->pose_total[5] = sn * T0 + cs * T1 + ty;
  st->pose_last[0] = cs; st->pose_last[1] = -sn; st->pose_last[2] = sn;
  st->pose_last[3] = cs; st->pose_last[4] = tx; st->pose_last[5] = ty;
  st->error = mean_error; st->mean_d2 = tot[9] * inv; st->inliers = (int)(cnt + 0.5);
  const int it = st->iterations + 1;
  st->iterations = it;                                               // > applied: the increment is pending
  const bool converged = fabs(st->prev_error - mean_error) < a.tolerance;   // icp.py:49-50
  st->prev_error = mean_error;                                               // icp.py:51
  if (converged || it >= a.max_iterations) st->done = 1;
}

// apply the increment the last update left pending (icp.py:45), so that src64 is the final cloud
__global__ void __launch_bounds__(256) s2m_finish_kernel(double* src64, int n, b200icp_s2m_state* st,
                                                         unsigned* scratch) {
  const bool pending = st->applied < st->iterations;
  if (pending) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
      const double2 s = apply_pending(st, make_double2(src64[2 * i], src64[2 * i + 1]));
      src64[2 * i] = s.x; src64[2 * i + 1] = s.y;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned ticket = atomicAdd(scratch + kTicketFinish, 1u);
    if (ticket == gridDim.x - 1) {
      scratch[kTicketFinish] = 0u;
      if (pending) st->applied = st->iterations;
    }
  }
}

int update_ctas(int n) {
  const int c = (n + kUpdateThreads - 1) / kUpdateThreads;
  return c < 1 ? 1 : (c > kMaxUpdateCtas ? kMaxUpdateCtas : c);
}

}  // namespace

extern "C" {

int b200icp_s2m_chunk(void) { return kChunk; }

int64_t b200icp_s2m_padded_chunks(int64_t m) {
  if (m < 1) return -1;
  const int64_t c = (m + kChunk - 1) / kChunk;
  return (c + kSuper - 1) / kSuper * kSuper;
}

int64_t b200icp_s2m_scratch_bytes(int32_t n_scan) {
  if (n_scan < 1) return -1;
  return (int64_t)kScratchHeader * 4 + (int64_t)kMaxUpdateCtas * 12 * 8;
}

int64_t b200icp_s2m_inbox_bytes(int32_t n_scan, int32_t world) {
  if (n_scan < 1 || world < 1 || world > kMaxWorld) return -1;
  return (int64_t)2 * world * n_scan * (int64_t)sizeof(b200icp_s2m_record) + (int64_t)(2 * world + 1) * 8;
}

int64_t b200icp_s2m_prepare_workspace_bytes(int64_t m) {
  if (m < 1 || m > 0x7fffffffLL) return -1;
  return sort_layout(m).total;
}

int b200icp_s2m_prepare_map(const b200icp_s2m_shard* shard, void* workspace, int64_t workspace_bytes,
                            void* stream) {
  if (!shard || !shard->points || !shard->chunk_circle || !shard->super_circle)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_prepare_map: NULL pointer");
  if (shard->m < 1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_prepare_map: empty shard");
  if (shard->dtype != B200ICP_F32 && shard->dtype != B200ICP_F64)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_prepare_map: bad dtype");
  if ((shard->sorted_points == nullptr) != (shard->order == nullptr))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_prepare_map: sorted_points and order go together");
  const int64_t n_chunks = (shard->m + kChunk - 1) / kChunk;
  const int64_t padded = b200icp_s2m_padded_chunks(shard->m);
  if (padded > (1LL << 24)) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "s2m_prepare_map: shard too large");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const void* scanned = shard->points;
  if (shard->sorted_points) {                   // Morton order (see above)
    if (shard->m > 0x7fffffffLL) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "s2m_prepare_map: spatial sort needs m < 2^31");
    const SortWs w = sort_layout(shard->m);
    if (!workspace || workspace_bytes < w.total) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_prepare_map: workspace too small");
    unsigned char* base = reinterpret_cast<unsigned char*>(workspace);
    unsigned long long* box = reinterpret_cast<unsigned long long*>(base + w.box);
    unsigned* keys_in = reinterpret_cast<unsigned*>(base + w.keys_in);
    unsigned* keys_out = reinterpret_cast<unsigned*>(base + w.keys_out);
    int32_t* idx_in = reinterpret_cast<int32_t*>(base + w.idx_in);
    if (cudaMemsetAsync(box, 0xff, 16, st) != cudaSuccess || cudaMemsetAsync(box + 2, 0, 16, st) != cudaSuccess)
      return check_launch("cudaMemsetAsync");
    const unsigned blocks = (unsigned)((shard->m + 255) / 256);
    s2m_bbox_kernel<<<blocks < 1184u ? blocks : 1184u, 256, 0, st>>>(shard->points, shard->dtype, shard->m, box);
    s2m_morton_kernel<<<blocks, 256, 0, st>>>(shard->points, shard->dtype, shard->m, box, keys_in, idx_in);
    size_t cub_bytes = w.cub_bytes;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(base + w.cub, cub_bytes, keys_in, keys_out, idx_in, shard->order,
                                                    (int)shard->m, 0, 32, st);
    if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "%s", cudaGetErrorString(e));
    s2m_gather_kernel<<<blocks, 256, 0, st>>>(shard->points, shard->dtype, shard->m, shard->order, shard->sorted_points);
    int rc = check_launch("s2m spatial sort");
    if (rc) return rc;
    scanned = shard->sorted_points;
  }
  s2m_prepare_kernel<<<(unsigned)padded, 256, 0, st>>>(scanned, shard->dtype, shard->m, (int)n_chunks,
                                                       shard->chunk_circle);
  int rc = check_launch("s2m_prepare_kernel");
  if (rc) return rc;
  s2m_super_kernel<<<(unsigned)(padded / kSuper), 32, 0, st>>>(shard->chunk_circle, shard->super_circle);
  return check_launch("s2m_super_kernel");
}

int b200icp_s2m_init(const void* scan, int32_t dtype, int32_t n, const double* init_pose,
                     double* src64, double* prev_nn, b200icp_s2m_state* state, void* stream) {
  if (!scan || !src64 || !state || n < 1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_init: bad arguments");
  if (dtype != B200ICP_F32 && dtype != B200ICP_F64) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_init: bad dtype");
  s2m_init_kernel<<<(n + 255) / 256, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      scan, dtype, n, init_pose, src64, prev_nn, state);
  return check_launch("s2m_init_kernel");
}

int b200icp_s2m_search(const b200icp_s2m_shard* shard, const b200icp_s2m_tables* tables, double* src64,
                       const double* prev_nn, int32_t n, b200icp_s2m_record* records,
                       void* const* peers, int32_t world, int32_t rank, b200icp_s2m_state* state,
                       void* scratch, void* stream) {
  if (!shard || !tables || !src64 || !state || !scratch || n < 1)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_search: bad arguments");
  if (!records && !peers) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_search: needs records or peers");
  if (peers && (world < 1 || world > kMaxWorld || rank < 0 || rank >= world))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_search: bad world / rank");
  if (!tables->chunk_circle || !tables->super_circle || tables->n_chunks_total % kSuper ||
      tables->first_local_chunk % kSuper || tables->n_local_chunks % kSuper ||
      tables->first_local_chunk + tables->n_local_chunks > tables->n_chunks_total ||
      (int64_t)tables->n_local_chunks != b200icp_s2m_padded_chunks(shard->m))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_search: inconsistent circle tables");
  SearchArgs a;
  if ((shard->sorted_points == nullptr) != (shard->order == nullptr))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_search: sorted_points and order go together");
  a.points = shard->sorted_points ? shard->sorted_points : shard->points; a.order = shard->order;
  a.m = shard->m; a.global_offset = shard->global_offset; a.dtype = shard->dtype;
  a.chunk_circle = tables->chunk_circle; a.super_circle = tables->super_circle;
  a.n_chunks_total = tables->n_chunks_total; a.first_local_chunk = tables->first_local_chunk;
  a.n_local_chunks = tables->n_local_chunks;
  a.src64 = src64; a.prev_nn = prev_nn; a.n = n; a.records = records; a.peers = peers;
  a.world = world; a.rank = rank; a.state = state; a.scratch = reinterpret_cast<unsigned*>(scratch);
  s2m_search_kernel<<<(n + kSearchWarps - 1) / kSearchWarps, kSearchWarps * 32, 0,
                      reinterpret_cast<cudaStream_t>(stream)>>>(a);
  return check_launch("s2m_search_kernel");
}

int b200icp_s2m_update(const b200icp_s2m_record* records_all, void* inbox, int32_t n_ranks, const double* src64,
                       double* prev_nn, int32_t n, int32_t max_iterations, double tolerance,
                       double max_corr_dist, int32_t* idx_out, b200icp_s2m_state* state, void* scratch,
                       void* stream) {
  if ((!records_all && !inbox) || !src64 || !prev_nn || !state || !scratch || n < 1 || n_ranks < 1 || n_ranks > kMaxWorld)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_update: bad arguments");
  UpdateArgs a;
  a.records_all = records_all; a.inbox = inbox; a.n_ranks = n_ranks; a.src64 = src64; a.prev_nn = prev_nn;
  a.n = n; a.max_iterations = max_iterations; a.tolerance = tolerance; a.max_corr_dist = max_corr_dist;
  a.idx_out = idx_out; a.state = state; a.scratch = reinterpret_cast<unsigned*>(scratch);
  s2m_update_kernel<<<update_ctas(n), kUpdateThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a);
  return check_launch("s2m_update_kernel");
}

int b200icp_s2m_finish(double* src64, int32_t n, b200icp_s2m_state* state, void* scratch, void* stream) {
  if (!src64 || !state || !scratch || n < 1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "s2m_finish: bad arguments");
  s2m_finish_kernel<<<(n + 255) / 256, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      src64, n, state, reinterpret_cast<unsigned*>(scratch));
  return check_launch("s2m_finish_kernel");
}

int b200icp_peer_alloc(int64_t bytes, void** ptr_out, void* handle_out) {
  if (bytes < 1 || !ptr_out || !handle_out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "peer_alloc: bad arguments");
  void* p = nullptr;
  if (cudaMalloc(&p, (size_t)bytes) != cudaSuccess) return check_launch("cudaMalloc");
  if (cudaMemset(p, 0, (size_t)bytes) != cudaSuccess) return check_launch("cudaMemset");
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, p) != cudaSuccess) { cudaFree(p); return check_launch("cudaIpcGetMemHandle"); }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  memcpy(handle_out, &h, 64);
  *ptr_out = p;
  return B200ICP_OK;
}

int b200icp_peer_open(const void* handle, void** ptr_out) {
  if (!handle || !ptr_out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "peer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  void* p = nullptr;
  if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) return check_launch("cudaIpcOpenMemHandle");
  *ptr_out = p;
  return B200ICP_OK;
}

int b200icp_peer_close(void* ptr) {
  if (ptr && cudaIpcCloseMemHandle(ptr) != cudaSuccess) return check_launch("cudaIpcCloseMemHandle");
  return B200ICP_OK;
}

int b200icp_peer_free(void* ptr) {
  if (ptr && cudaFree(ptr) != cudaSuccess) return check_launch("cudaFree");
  return B200ICP_OK;
}

#if S2M_TIMING
// debug builds only (tools/build_variant.py ... -DS2M_TIMING=1): read and clear the phase counters
int b200icp_s2m_debug_clocks(unsigned long long* out8) {
  unsigned long long zero[8] = {};
  if (cudaMemcpyFromSymbol(out8, g_s2m_clk, sizeof(zero)) != cudaSuccess) return B200ICP_ERR_CUDA;
  if (cudaMemcpyToSymbol(g_s2m_clk, zero, sizeof(zero)) != cudaSuccess) return B200ICP_ERR_CUDA;
  return B200ICP_OK;
}
#endif

}  // extern "C"
