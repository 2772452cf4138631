// occupancy.cu -- occupancy-grid ray casting on the device (sm_100a), SURVEY.md 8(f) rank 4.
//
// Replaces update_occupancy_map (duc/ICP_LIDAR/process.py:114-177, same body at
// duc/ICP_LIDAR/slam_offline.py:174-236) with its bresenham_line (process.py:86-112), and the
// cell-probability point filter filter_new_points_by_occupancy / prune_global_map
// (process.py:203-249).  Results are bit-identical to the reference: float32 probabilities,
// uint8 grey levels, kept-point order.
//
// The update is ORDER DEPENDENT: a ray multiplies free cells by p_free_dec until it meets a
// cell >= 0.65 (which ends the ray before its end cell is raised), the end cell is raised by
// p_occ_inc, and adjacent beams share most of their first ~50 cells.  Exactness therefore
// fixes the order of the beams of one map; what is parallel is
//   (1) the geometry: the threads of the CTA convert end points to cells, and 12 producer warps
//       expand the rays into cell lists (closed form of the reference's Bresenham walk, no serial
//       stepping) in a shared-memory ring, ahead of the ordered loop;
//   (2) the cells of one ray: distinct by construction, so the ordered warp reads all of them at
//       once (128 per trip) from a shared-memory tile of the map, finds the first blocking cell with
//       a vote and writes the cells before it -- one shared-memory round trip per ray instead of
//       one global-memory round trip per cell;
//   (3) the grey-level rendering: only the cells that leave the window per frame, the last window
//       once per launch, all threads;
//   (4) independent maps (recordings / robots): one CTA per map, any number of frames per
//       launch, applied in order.
// DESIGN.md 4.5d has the measurements and what was tried and rejected.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>

#include "common.cuh"
#include "compact.cuh"

namespace {

constexpr int kOccThreads = 512;
constexpr int kOccUnroll = 5;                 // on-map fallback: 5 x 32 cells per trip
constexpr int kOccTileCells = 54 * 1024;      // float32 map cells held in shared memory (216 KB)
constexpr int kOccTileMargin = 8;             // cells added around a new tile when they fit
constexpr int kOccSmemBytes = 227 * 1024;     // tile + ring of per-ray cell lists
constexpr int kOccGroup = 512;                // rays whose end cells are resident at once
constexpr int kOccMaxSlots = 16;              // ring slots (rays expanded ahead of the ordered loop)
constexpr int kOccProducers = 12;             // warps expanding rays into the ring

// int(): truncation toward zero (Python's int(float)); callers test finiteness first
__device__ __forceinline__ long long py_int(double v) { return (long long)v; }

struct OccWindow {
  long long x1, y1;       // window origin in the map (process.py:130-131)
  long long rx, ry;       // robot cell relative to the window (:140-141)
  int width, height;      // window size after Python's slice clamping (:134-138)
};

// len(range(*slice(a, b).indices(n))) for a >= 0: a negative stop counts from the end
__device__ __forceinline__ int slice_len(long long a, long long b, int n) {
  if (b < 0) { b += n; if (b < 0) b = 0; }
  if (b > n) b = n;
  if (a > n) a = n;
  return b > a ? (int)(b - a) : 0;
}

__device__ __forceinline__ OccWindow occ_window(const b200icp_occ_grid& g, double robot_x, double robot_y) {
  OccWindow wdw;
  const long long rxp = py_int(__dadd_rn(g.center_x, __ddiv_rn(robot_x, g.resolution)));   // :128
  const long long ryp = py_int(__dsub_rn(g.center_y, __ddiv_rn(robot_y, g.resolution)));   // :129
  wdw.x1 = max(0ll, rxp - g.area);
  wdw.y1 = max(0ll, ryp - g.area);
  const long long x2 = min((long long)g.w, rxp + g.area), y2 = min((long long)g.h, ryp + g.area);
  wdw.width = slice_len(wdw.x1, x2, g.w);
  wdw.height = slice_len(wdw.y1, y2, g.h);
  wdw.rx = rxp - wdw.x1;
  wdw.ry = ryp - wdw.y1;
  return wdw;
}

// Cell k of bresenham_line(rx, ry, px, py) (process.py:86-112).  With the error term doubled it
// stays in [0, 2*major), so after k steps along the major axis the minor axis has advanced
// floor((2*k*minor + major - 1) / (2*major)) times.
__device__ __forceinline__ void bres_cell(int rx, int ry, int px, int py, int k, int& x, int& y) {
  const int dx = abs(px - rx), dy = abs(py - ry);
  const int sx = rx > px ? -1 : 1, sy = ry > py ? -1 : 1;
  if (dx > dy) {
    x = rx + sx * k;
    y = ry + sy * (int)((2u * (unsigned)k * (unsigned)dy + (unsigned)dx - 1u) / (2u * (unsigned)dx));
  } else {
    y = ry + sy * k;
    x = dy == 0 ? rx : rx + sx * (int)((2u * (unsigned)k * (unsigned)dx + (unsigned)dy - 1u) / (2u * (unsigned)dy));
  }
}

template <typename T>
__device__ __forceinline__ double2 occ_load_point(const void* base, int64_t i) {
  const T* p = reinterpret_cast<const T*>(base) + 2 * i;
  return make_double2((double)p[0], (double)p[1]);
}

struct OccRect {          // half-open rectangle of map cells
  int x0, y0, x1, y1;
  __device__ __forceinline__ int w() const { return x1 - x0; }
  __device__ __forceinline__ int h() const { return y1 - y0; }
  __device__ __forceinline__ bool empty() const { return x1 <= x0 || y1 <= y0; }
  __device__ __forceinline__ bool contains(const OccRect& r) const {
    return r.x0 >= x0 && r.y0 >= y0 && r.x1 <= x1 && r.y1 <= y1;
  }
};

__device__ __forceinline__ OccRect rect_union(const OccRect& a, const OccRect& b) {
  return OccRect{min(a.x0, b.x0), min(a.y0, b.y0), max(a.x1, b.x1), max(a.y1, b.y1)};
}

// One ray, all cells at once (see the header comment): `mem` is the shared-memory tile or the map
// itself, off_of(k) the cell of step k in it (-1 = outside the window, skipped).  Up to 160 cells
// per trip; `first` = pre-loaded offsets of the first trip.
template <typename OffFn>
__device__ __forceinline__ void occ_cast_ray(float* mem, int L, int lane, float thr_up, float dec, float inc,
                                             OffFn off_of) {
  bool stopped = false;
  for (int k0 = 0; k0 <= L && !stopped; k0 += 32 * kOccUnroll) {
    int off[kOccUnroll];
    float v[kOccUnroll];
#pragma unroll
    for (int u = 0; u < kOccUnroll; ++u) {
      const int k = k0 + u * 32 + lane;
      off[u] = k <= L ? off_of(k) : -1;
    }
#pragma unroll
    for (int u = 0; u < kOccUnroll; ++u) v[u] = off[u] >= 0 ? mem[off[u]] : 0.0f;
#pragma unroll
    for (int u = 0; u < kOccUnroll; ++u) {
      const int k = k0 + u * 32 + lane;
      const bool free_cell = off[u] >= 0 && k < L;
      const unsigned hit = __ballot_sync(kFull, free_cell && v[u] >= thr_up);                 // :165
      if (!stopped) {
        const int first = hit ? __ffs(hit) - 1 : 32;
        if (free_cell && lane < first) {
          const float nv = __fmul_rn(v[u], dec);                                                   // :167
          mem[off[u]] = nv > 0.0f ? nv : 0.0f;                                                    // max(0.0, .) as Python evaluates it
        }
        if (hit) stopped = true;                                                                   // :166 break
        else if (k == L && off[u] >= 0) {                                                          // :162-163
          const float nv = __fadd_rn(v[u], inc);
          mem[off[u]] = nv < 1.0f ? nv : 1.0f;                                                     // min(1.0, .)
        }
      }
    }
  }
  __syncwarp();        // orders this ray's stores before the next ray's loads (other lanes)
}

// grey levels of a rectangle of map cells (process.py:172-176), byte-coalesced.  Cells held by
// the shared-memory tile (trect, pitch tp) are read there -- the tile may be newer than the map.
// No __restrict__: the probabilities were written earlier in this kernel (no LDG.NC).
__device__ __forceinline__ void occ_render_rect(const float* probs, uint8_t* image, int W, OccRect r,
                                                const float* tile, OccRect trect, int tp,
                                                int warp, int lane, int n_warps) {
  if (r.empty()) return;
  if (r.w() < 32) {                       // thin strip (the window moved by a cell or two): one thread per cell
    const int rw = r.w(), cells = rw * r.h();
    for (int c = warp * 32 + lane; c < cells; c += 32 * n_warps) {
      const int yy = c / rw, x = r.x0 + (c - yy * rw), y = r.y0 + yy;
      const bool in = y >= trect.y0 && y < trect.y1 && x >= trect.x0 && x < trect.x1;
      const float v = in ? tile[(y - trect.y0) * tp + (x - trect.x0)] : probs[(size_t)y * W + x];
      const uint8_t u8 = (uint8_t)(int)__fmul_rn(__fsub_rn(1.0f, v), 255.0f);
      uint8_t* dst = image + ((size_t)y * W + x) * 3;
      dst[0] = u8; dst[1] = u8; dst[2] = u8;
    }
    return;
  }
  const int bytes = 3 * r.w();
  for (int y = r.y0 + warp; y < r.y1; y += n_warps) {
    const float* src = probs + (size_t)y * W;
    const bool row_in = y >= trect.y0 && y < trect.y1;
    const float* trow = tile + (y - trect.y0) * tp - trect.x0;
    uint8_t* dst = image + ((size_t)y * W + r.x0) * 3;
    for (int j0 = lane; j0 < bytes; j0 += 128) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int x = r.x0 + (j0 + 32 * u) / 3;
        v[u] = j0 + 32 * u < bytes ? ((row_in && x >= trect.x0 && x < trect.x1) ? trow[x] : src[x]) : 0.0f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (j0 + 32 * u < bytes) dst[j0 + 32 * u] = (uint8_t)(int)__fmul_rn(__fsub_rn(1.0f, v[u]), 255.0f);
    }
  }
}

// shared-memory pitch of a tile of w columns: odd and = 3 or 5 (mod 8), so that vertical rays are
// conflict-free and exact diagonals at most 4-way conflicted
__device__ __forceinline__ int occ_tile_pitch(int w) {
  int p = w | 1;
  while ((p & 7) != 3 && (p & 7) != 5) p += 2;
  return p;
}

// ---- shared-memory primitives with 32-bit addresses (the ordered loop is one warp deep: every
// instruction on its path counts, so no generic-address arithmetic there) ----------------------
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory");
}
__device__ __forceinline__ int4 lds_v4(uint32_t a) {
  int4 v;
  asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ int lds_volatile(uint32_t a) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts_volatile(uint32_t a, int v) {
  asm volatile("st.volatile.shared.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// One CTA per map; frames in order; see the header comment.
//
// Shared memory (32-bit words):
//   tile[kOccTileCells]   a rectangle of the map -- the cells the rays of a run can touch -- kept
//                         across runs / groups / frames while the next rays stay inside it; [+4]: a
//                         dummy cell (0.0) that absorbs the lanes and list entries with no cell
//   ends[kOccGroup]       end cell of every ray of the group, window coordinates, x | y << 16
//                         (0xffffffff: the point is outside the window -> ray skipped)
//   ctrl[32]              ready[16] tickets, done ticket, group bounding box
//   ring[K][4 + stride]   cell lists of the K rays in flight: header {L, end cell address}, then
//                         the shared-memory address of every free cell (k < L), dummy-padded to 4
// Warp 0 is the ORDERED loop: it takes rays in order from the ring, reads all cells of a ray at
// once, votes, writes.  Warps 1..15 are producers: they expand rays (closed-form Bresenham) into
// ring slots ahead of warp 0, so none of the geometry is on the ordered path.
// A ray has at most area + 1 cells unless the robot is more than `area` cells outside the map on
// the low side (Python's negative slice stop then makes the window nearly the whole map,
// process.py:132-136); such rays (L >= stride) and rays whose bounding box exceeds the tile are
// cast directly on the map in global memory, cells evaluated on the fly.
__global__ void __launch_bounds__(kOccThreads) occ_update_kernel(b200icp_occ_grid g, const void* points,
                                                                 int dtype, const int32_t* len,
                                                                 const double* robot_xy, int n_frames,
                                                                 int pitch, int K, int stride) {
  extern __shared__ int occ_smem[];
  float* tile = reinterpret_cast<float*>(occ_smem);
  unsigned* ends = reinterpret_cast<unsigned*>(occ_smem) + kOccTileCells + 4;
  int* ctrl = occ_smem + kOccTileCells + 4 + kOccGroup;
  int* ring = ctrl + 32;
  const int slot_words = stride + 4;
  const uint32_t tile_sa = (uint32_t)__cvta_generic_to_shared(tile);
  const uint32_t dummy_sa = tile_sa + 4u * kOccTileCells;
  const uint32_t ctrl_sa = (uint32_t)__cvta_generic_to_shared(ctrl);
  const uint32_t ring_sa = (uint32_t)__cvta_generic_to_shared(ring);
  const uint32_t done_sa = ctrl_sa + 4u * 16;
  const int map = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kOccThreads / 32;
  float* probs = g.probs + (size_t)map * g.h * g.w;
  uint8_t* image = g.image ? g.image + (size_t)map * g.h * g.w * 3 : nullptr;
  const float thr_up = g.threshold_up, dec = g.p_free_dec, inc = g.p_occ_inc;
  const int W = g.w;

#ifdef B200ICP_OCC_PROFILE
  long long prof[6] = {0, 0, 0, 0, 0, 0}, prof_last = clock64();
  int prof_loads = 0, prof_runs = 0;
#define OCC_TICK(i) do { const long long now_ = clock64(); prof[i] += now_ - prof_last; prof_last = now_; } while (0)
#else
#define OCC_TICK(i) do { } while (0)
#endif
  OccRect trect{0, 0, 0, 0};          // map rectangle held by the tile (uniform across the CTA)
  bool tile_dirty = false;
  OccRect shown{0, 0, 0, 0};          // window whose picture is still to be rendered
  int tbase = 0;                      // tickets handed out so far (uniform)

  if (tid < 32) ctrl[tid] = 0;
  if (tid == 0) tile[kOccTileCells] = 0.0f;
  for (int i = tid; i < K * slot_words; i += kOccThreads) ring[i] = (int)dummy_sa;   // stale entries stay valid addresses
  __syncthreads();

  auto flush_tile = [&]() {           // tile -> map (all threads), keeps the tile valid
    if (tile_dirty) {
      const int tw = trect.w(), tp = occ_tile_pitch(tw), th = trect.h();
      for (int y0 = warp; y0 < th; y0 += 2 * kWarps)             // 2 rows x 4 column groups per trip
        for (int x0 = lane; x0 < tw; x0 += 128) {
          float v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int y = y0 + (u >> 2) * kWarps, x = x0 + 32 * (u & 3);
            v[u] = (y < th && x < tw) ? lds_f32(tile_sa + 4u * (unsigned)(y * tp + x)) : 0.0f;
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int y = y0 + (u >> 2) * kWarps, x = x0 + 32 * (u & 3);
            if (y < th && x < tw) probs[(size_t)(trect.y0 + y) * W + trect.x0 + x] = v[u];
          }
        }
      tile_dirty = false;
    }
    __syncthreads();
  };
  // map -> tile (all threads); caller has flushed.  Asynchronous 4-byte copies (LDGSTS): every
  // thread keeps its whole share of the rectangle in flight, no register staging, any alignment.
  auto load_tile = [&](const OccRect& r) {
    trect = r;
    const int tw = r.w(), tp = occ_tile_pitch(tw), th = r.h();
    for (int y = warp; y < th; y += kWarps) {
      const float* src = probs + (size_t)(r.y0 + y) * W + r.x0;
      const uint32_t dst = tile_sa + 4u * (unsigned)(y * tp);
      for (int x = lane; x < tw; x += 32)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * (unsigned)x), "l"(src + x) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
  };

  for (int f = 0; f < n_frames; ++f) {
    const int64_t fr = (int64_t)map * n_frames + f;
    const int n = min(len ? len[fr] : pitch, pitch);
    if (n <= 0) continue;                                           // process.py:116-117
    const OccWindow wdw = occ_window(g, robot_xy[2 * fr], robot_xy[2 * fr + 1]);
    const int rx = (int)max(-(1ll << 30), min(1ll << 30, wdw.rx));
    const int ry = (int)max(-(1ll << 30), min(1ll << 30, wdw.ry));
    const int wx1 = (int)min(wdw.x1, (long long)g.w), wy1 = (int)min(wdw.y1, (long long)g.h);
    const double x1d = (double)wdw.x1, y1d = (double)wdw.y1;
    const OccRect wrect{wx1, wy1, wx1 + wdw.width, wy1 + wdw.height};

    // the picture of the previous window: cells that leave the window are final until a later
    // window covers them again, so only they are rendered now (the rest with the last frame)
    if (image && !shown.empty() && !(shown.x0 == wrect.x0 && shown.y0 == wrect.y0 && shown.x1 == wrect.x1 && shown.y1 == wrect.y1)) {
      const int ttp = occ_tile_pitch(trect.w());
      const int oy0 = max(shown.y0, wrect.y0), oy1 = min(shown.y1, wrect.y1);      // rows shared with the new window
      if (wrect.empty() || oy0 >= oy1 || max(shown.x0, wrect.x0) >= min(shown.x1, wrect.x1)) {
        occ_render_rect(probs, image, W, shown, tile, trect, ttp, warp, lane, kWarps);
      } else {
        occ_render_rect(probs, image, W, OccRect{shown.x0, shown.y0, shown.x1, oy0}, tile, trect, ttp, warp, lane, kWarps);
        occ_render_rect(probs, image, W, OccRect{shown.x0, oy1, shown.x1, shown.y1}, tile, trect, ttp, warp, lane, kWarps);
        occ_render_rect(probs, image, W, OccRect{shown.x0, oy0, max(shown.x0, wrect.x0), oy1}, tile, trect, ttp, warp, lane, kWarps);
        occ_render_rect(probs, image, W, OccRect{min(shown.x1, wrect.x1), oy0, shown.x1, oy1}, tile, trect, ttp, warp, lane, kWarps);
      }
    }
    shown = wrect;
    OCC_TICK(4);
    if (wrect.empty()) continue;                                    // no point can fall into it (:150)

    // the window coordinates of the robot cell, clipped to the window (rays start there)
    const int rcx = min(max(rx, 0), wdw.width - 1), rcy = min(max(ry, 0), wdw.height - 1);
    auto ray_len = [&](unsigned e) { return max(abs((int)(e & 0xffffu) - rx), abs((int)(e >> 16) - ry)); };
    auto ray_rect = [&](unsigned e) {        // map rectangle of a ray: robot cell and end cell
      const int ex = (int)(e & 0xffffu), ey = (int)(e >> 16);
      return OccRect{min(rcx, ex) + wx1, min(rcy, ey) + wy1, max(rcx, ex) + 1 + wx1, max(rcy, ey) + 1 + wy1};
    };
    auto fits = [&](const OccRect& r) { return occ_tile_pitch(r.w()) * r.h() <= kOccTileCells; };

    for (int g0 = 0; g0 < n; g0 += kOccGroup) {
      const int ng = min(kOccGroup, n - g0);
      // ---- geometry: end cell of every ray of the group, and their bounding box ---------------
      if (tid < 8) ctrl[20 + tid] = (tid & 1) ? -1 : 0x7fffffff;   // min x, max x, min y, max y, listed-only flag ...
      __syncthreads();
      {
        int mnx = 0x7fffffff, mxx = -1, mny = 0x7fffffff, mxy = -1, unlisted = 0;
        for (int b = tid; b < ng; b += kOccThreads) {
          const int64_t i = fr * pitch + g0 + b;
          const double2 q = dtype == B200ICP_F64 ? occ_load_point<double>(points, i) : occ_load_point<float>(points, i);
          const double fx = __dsub_rn(__dadd_rn(g.center_x, __ddiv_rn(q.x, g.resolution)), x1d);   // :147
          const double fy = __dsub_rn(__dsub_rn(g.center_y, __ddiv_rn(q.y, g.resolution)), y1d);   // :148
          unsigned e = 0xffffffffu;
          if (isfinite(fx) && isfinite(fy)) {
            const long long px = py_int(fx), py = py_int(fy);
            if (0 <= px && px < wdw.width && 0 <= py && py < wdw.height) {                          // :150
              e = (unsigned)px | ((unsigned)py << 16);
              mnx = min(mnx, (int)px); mxx = max(mxx, (int)px); mny = min(mny, (int)py); mxy = max(mxy, (int)py);
              if (K < 2 || ray_len(e) >= stride) unlisted = 1;
            }
          }
          ends[b] = e;
        }
        mnx = __reduce_min_sync(kFull, mnx); mxx = __reduce_max_sync(kFull, mxx);
        mny = __reduce_min_sync(kFull, mny); mxy = __reduce_max_sync(kFull, mxy);
        unlisted = __reduce_max_sync(kFull, unlisted);
        if (lane == 0 && mxx >= 0) {
          atomicMin(&ctrl[20], mnx); atomicMax(&ctrl[21], mxx); atomicMin(&ctrl[22], mny); atomicMax(&ctrl[23], mxy);
          if (unlisted) atomicMax(&ctrl[25], 1);
        }
      }
      __syncthreads();
      OCC_TICK(0);
      const int gx0 = ctrl[20], gx1 = ctrl[21], gy0 = ctrl[22], gy1 = ctrl[23];
      const bool any_unlisted = ctrl[25] > 0;
      if (gx1 < 0) continue;                                        // no ray in this group
      const OccRect gbb{min(rcx, gx0) + wx1, min(rcy, gy0) + wy1, max(rcx, gx1) + 1 + wx1, max(rcy, gy1) + 1 + wy1};

      // ---- runs of consecutive rays that share one tile (every thread takes the same decisions) --
      int s = 0;
      while (s < ng) {
        int e = s;
        bool on_map = false;
        if (!any_unlisted && trect.contains(gbb)) {
          e = ng;                                                   // the tile already holds the whole group
        } else if (!any_unlisted && s == 0 && fits(gbb)) {
          OccRect bb = gbb;                                         // one new tile for the whole group,
          const OccRect lim{max(wrect.x0 - kOccTileMargin, 0), max(wrect.y0 - kOccTileMargin, 0),
                            min(wrect.x1 + kOccTileMargin, g.w), min(wrect.y1 + kOccTileMargin, g.h)};
          for (int m = 64; m > 0; m >>= 1) {                        // grown around the window as far as it fits:
            const OccRect gr{max(bb.x0 - m, lim.x0), max(bb.y0 - m, lim.y0),       // the next frames stay inside it
                             min(bb.x1 + m, lim.x1), min(bb.y1 + m, lim.y1)};
            if (fits(gr)) bb = gr;
          }
          flush_tile();
          load_tile(bb);
#ifdef B200ICP_OCC_PROFILE
          ++prof_loads;
#endif
          e = ng;
        } else {                                                    // ray by ray
          const unsigned es = ends[s];
          if (es == 0xffffffffu) { ++s; continue; }
          const bool listed_s = K >= 2 && ray_len(es) < stride;
          if (listed_s && trect.contains(ray_rect(es))) {
            e = s + 1;
            while (e < ng) {
              const unsigned ee = ends[e];
              if (ee != 0xffffffffu && !(ray_len(ee) < stride && trect.contains(ray_rect(ee)))) break;
              ++e;
            }
          } else if (!listed_s || !fits(ray_rect(es))) {
            on_map = true;                                          // cast on the map itself
            e = s + 1;
          } else {
            OccRect bb = ray_rect(es);
            e = s + 1;
            while (e < ng) {
              const unsigned ee = ends[e];
              if (ee != 0xffffffffu) {
                if (ray_len(ee) >= stride) break;
                const OccRect u = rect_union(bb, ray_rect(ee));
                if (!fits(u)) break;
                bb = u;
              }
              ++e;
            }
            flush_tile();
            load_tile(bb);
#ifdef B200ICP_OCC_PROFILE
            ++prof_loads;
#endif
          }
        }
        OCC_TICK(1);
#ifdef B200ICP_OCC_PROFILE
        ++prof_runs;
#endif
        if (on_map) {
          flush_tile();
          trect = OccRect{0, 0, 0, 0};
          if (warp == 0) {
            const unsigned es = ends[s];
            const int L = ray_len(es), px = (int)(es & 0xffffu), py = (int)(es >> 16);
            occ_cast_ray(probs, L, lane, thr_up, dec, inc, [&](int k) {
              int x, y;
              bres_cell(rx, ry, px, py, k, x, y);
              const bool in = 0 <= x && x < wdw.width && 0 <= y && y < wdw.height;                // :152
              return in ? (wy1 + y) * W + (wx1 + x) : -1;
            });
          }
          __syncthreads();
          OCC_TICK(5);
        } else {
          const int tp = occ_tile_pitch(trect.w()), tox = wx1 - trect.x0, toy = wy1 - trect.y0;
          if ((warp & 3) != 0) {
            // ---- producers (warps 1-3, 5-7, 9-11, 13-15; warps 4, 8, 12 stay out of the way so that
            // the ordered loop has its scheduler to itself): ray b -> ring slot, ahead of warp 0 ----
            const int pidx = warp - 1 - (warp >> 2);
            int slot = (tbase + pidx) % K;
            for (int b = s + pidx; b < e; b += kOccProducers) {
              const int ticket = tbase + (b - s);
              if (lane == 0)
                while (lds_volatile(done_sa) - (ticket - K + 1) < 0) __nanosleep(64);   // slot consumed?
              __syncwarp();
              int* sl = ring + (size_t)slot * slot_words;
              const unsigned eb = ends[b];
              if (eb == 0xffffffffu) {
                if (lane == 0) sl[0] = -1;
              } else {
                const int px = (int)(eb & 0xffffu), py = (int)(eb >> 16);
                const int dx = abs(px - rx), dy = abs(py - ry), L = max(dx, dy), mn = min(dx, dy);
                const int sx = rx > px ? -1 : 1, sy = ry > py ? -1 : 1;
                const bool xmajor = dx > dy;                                  // process.py:93
                const unsigned dd = 2u * (unsigned)max(L, 1), magic = 0xffffffffu / dd;
                const int Lp = max((L + 3) & ~3, 128);                        // the first trip reads 128 entries
                for (int k = lane; k < Lp; k += 32) {
                  int a = (int)dummy_sa;
                  if (k < L) {
                    // minor-axis steps after k major steps: floor((2 k mn + L - 1) / (2 L))
                    const unsigned num = 2u * (unsigned)k * (unsigned)mn + (unsigned)L - 1u;
                    unsigned q = __umulhi(num, magic), r = num - q * dd;
                    while (r >= dd) { ++q; r -= dd; }
                    const int x = xmajor ? rx + sx * k : rx + sx * (int)q;
                    const int y = xmajor ? ry + sy * (int)q : ry + sy * k;
                    if (0 <= x && x < wdw.width && 0 <= y && y < wdw.height)                       // :152
                      a = (int)(tile_sa + 4u * (unsigned)((toy + y) * tp + (tox + x)));
                  }
                  sl[4 + k] = a;
                }
                if (lane == 0) {
                  sl[0] = L;
                  sl[1] = (int)(tile_sa + 4u * (unsigned)((toy + py) * tp + (tox + px)));
                }
              }
              __threadfence_block();
              __syncwarp();
              if (lane == 0) sts_volatile(ctrl_sa + 4u * slot, ticket + 1);
              slot += kOccProducers % K;      // K may be smaller than the producer count
              if (slot >= K) slot -= K;
            }
          } else if (warp == 0) {
            // ---- the ordered loop: lane l owns cells 4l .. 4l+3 of a 128-cell trip; the common
            // case -- no cell of the ray blocks -- is one vote and straight-line stores.  The list of
            // the next ray is fetched while the cells of the current one are in flight. -----------
            int slot = tbase % K;
            uint32_t sl = ring_sa + 4u * (unsigned)(slot * slot_words);
            while (lds_volatile(ctrl_sa + 4u * slot) != tbase + 1) { }
            int4 hdr = lds_v4(sl), o = lds_v4(sl + 16u + 16u * (unsigned)lane);
            for (int b = s; b < e; ++b) {
              const int ticket = tbase + (b - s);
              const int L = hdr.x;
              const uint32_t eo = L >= 0 ? (uint32_t)hdr.y : dummy_sa;
              const uint32_t cur_sl = sl;
              const float ev = lds_f32(eo);                                  // end cell: not on the free part
              float v0 = lds_f32((uint32_t)o.x), v1 = lds_f32((uint32_t)o.y);
              float v2 = lds_f32((uint32_t)o.z), v3 = lds_f32((uint32_t)o.w);
              int4 oc = o;
              if (b + 1 < e) {                                               // next ray's list
                ++slot; sl += 4u * (unsigned)slot_words;
                if (slot == K) { slot = 0; sl = ring_sa; }
#ifdef B200ICP_OCC_PROFILE
                const long long w0_ = clock64();
#endif
                while (lds_volatile(ctrl_sa + 4u * slot) != ticket + 2) { }
#ifdef B200ICP_OCC_PROFILE
                prof[2] += clock64() - w0_;
#endif
                hdr = lds_v4(sl);
                o = lds_v4(sl + 16u + 16u * (unsigned)lane);
              }
              if (L >= 0) {
                bool stopped = false;
                for (int k0 = 0; k0 < L; k0 += 128) {
                  if (k0 > 0) {                                              // rays longer than one trip
                    const int kl = k0 + 4 * lane;
                    oc = make_int4((int)dummy_sa, (int)dummy_sa, (int)dummy_sa, (int)dummy_sa);
                    if (kl < L) oc = lds_v4(cur_sl + 16u + 4u * (unsigned)kl);
                    v0 = lds_f32((uint32_t)oc.x); v1 = lds_f32((uint32_t)oc.y);
                    v2 = lds_f32((uint32_t)oc.z); v3 = lds_f32((uint32_t)oc.w);
                  }
                  const bool h0 = v0 >= thr_up, h1 = v1 >= thr_up, h2 = v2 >= thr_up, h3 = v3 >= thr_up;   // :165
                  int first = 4;                                            // cells of this lane to update
                  if (__any_sync(kFull, h0 | h1 | h2 | h3)) {          // :166 break
                    const int mine = h0 ? 0 : h1 ? 1 : h2 ? 2 : h3 ? 3 : 4;
                    const unsigned lanes = __ballot_sync(kFull, mine < 4);
                    const int fl = __ffs(lanes) - 1;                        // first blocking lane
                    first = lane < fl ? 4 : lane == fl ? mine : 0;
                    stopped = true;
                  }
                  float n0 = __fmul_rn(v0, dec), n1 = __fmul_rn(v1, dec), n2 = __fmul_rn(v2, dec), n3 = __fmul_rn(v3, dec);   // :167
                  n0 = n0 > 0.0f ? n0 : 0.0f; n1 = n1 > 0.0f ? n1 : 0.0f;    // max(0.0, .) as Python evaluates it
                  n2 = n2 > 0.0f ? n2 : 0.0f; n3 = n3 > 0.0f ? n3 : 0.0f;
                  if (first > 0) sts_f32((uint32_t)oc.x, n0);
                  if (first > 1) sts_f32((uint32_t)oc.y, n1);
                  if (first > 2) sts_f32((uint32_t)oc.z, n2);
                  if (first > 3) sts_f32((uint32_t)oc.w, n3);
                  if (stopped) break;
                }
                if (!stopped && lane == 0) {                                // :162-163
                  const float nv = __fadd_rn(ev, inc);
                  sts_f32(eo, nv < 1.0f ? nv : 1.0f);                       // min(1.0, .)
                }
              }
              __syncwarp();      // orders this ray's stores before the next ray's loads (other lanes)
              if (lane == 0) sts_volatile(done_sa, ticket + 1);
            }
            sts_f32(dummy_sa, 0.0f);
          }
          tbase += e - s;
          tile_dirty = true;
          __syncthreads();
          OCC_TICK(3);
        }
        s = e;
      }
    }
  }
  flush_tile();
  OCC_TICK(1);
  if (image) occ_render_rect(probs, image, W, shown, tile, OccRect{0, 0, 0, 0}, 1, warp, lane, kWarps);
  OCC_TICK(4);
#ifdef B200ICP_OCC_PROFILE
  if (tid == 0 && map == 0)
    printf("occ_prof cycles: geometry %lld, runs+tile_io %lld, chain_wait_for_producers %lld, chain_total %lld, render %lld, on_map %lld; tile loads %d, runs %d, frames %d\n",
           prof[0], prof[1], prof[2], prof[3], prof[4], prof[5], prof_loads, prof_runs, n_frames);
#endif
}

// ---- point filter (process.py:203-249): keep iff outside the grid or probs[py, px] >= thr -------
template <typename T>
struct OccKeep {
  const T* points;
  int cols;
  const float* probs;
  int h, w;
  double cx, cy, res;
  float thr;
  __device__ __forceinline__ bool operator()(int64_t i) const {
    const double fx = __dadd_rn(cx, __ddiv_rn((double)points[i * cols], res));          // :213
    const double fy = __dsub_rn(cy, __ddiv_rn((double)points[i * cols + 1], res));      // :214
    if (!(isfinite(fx) && isfinite(fy))) return true;
    const long long px = py_int(fx), py = py_int(fy);
    if (!(0 <= px && px < w && 0 <= py && py < h)) return true;                           // :216-218
    return !(probs[py * w + px] < thr);                                                   // :220-221
  }
};

struct KeptIndex {
  int64_t* out;
  __device__ __forceinline__ void operator()(int64_t dst, int64_t i) const { out[dst] = i; }
};

bool occ_grid_ok(const b200icp_occ_grid* g, const char* who) {
  const char* why = nullptr;
  if (!g) why = "grid is NULL";
  else if (!g->probs) why = "grid.probs is NULL";
  else if (g->h < 1 || g->w < 1 || g->h > 32768 || g->w > 32768) why = "grid.h / grid.w must be in [1, 32768]";
  else if (!(g->resolution > 0.0)) why = "grid.resolution must be > 0";
  else if (!(g->threshold_up > 0.0f)) why = "grid.threshold_up must be > 0";
  if (!why) return true;
  set_error(B200ICP_ERR_INVALID_ARGUMENT, "%s: %s", who, why);
  return false;
}

}  // namespace

extern "C" {

int b200icp_occ_update(const b200icp_occ_grid* grid, int32_t n_maps, const void* points, int32_t dtype,
                       const int32_t* len, const double* robot_xy, int32_t n_frames, int32_t pitch,
                       void* stream) {
  if (!occ_grid_ok(grid, "occ_update")) return B200ICP_ERR_INVALID_ARGUMENT;
  if (n_maps < 0 || n_frames < 0 || pitch < 0 || (!points && pitch > 0) || !robot_xy)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "occ_update: bad arguments");
  if (dtype != B200ICP_F32 && dtype != B200ICP_F64) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "occ_update: bad dtype");
  if (grid->area < 0 || grid->area > 10000) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "occ_update: area must be in [0, 10000]");
  if (n_maps == 0 || n_frames == 0 || pitch == 0) return B200ICP_OK;
  // ring of K cell lists behind the tile; a ray has <= area + 1 cells (int4 rows)
  int stride = (grid->area + 1 + 3) & ~3;
  if (stride < 128) stride = 128;                                  // the ordered loop reads 128 entries per trip
  const int avail = kOccSmemBytes / 4 - kOccTileCells - 4 - kOccGroup - 32;
  int K = avail / (stride + 4);
  if (K > kOccMaxSlots) K = kOccMaxSlots;
  if (K < 2) { K = 0; stride = 0; }                                // window too large for lists: rays are cast on the map
  const size_t smem = ((size_t)kOccTileCells + 4 + kOccGroup + 32 + (size_t)K * (stride + 4)) * sizeof(int);
  static thread_local int configured_device = -1;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "occ_update: cudaGetDevice: %s", cudaGetErrorString(e));
  if (configured_device != dev) {
    e = cudaFuncSetAttribute(occ_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kOccSmemBytes);
    if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "occ_update: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    configured_device = dev;
  }
  occ_update_kernel<<<n_maps, kOccThreads, smem, reinterpret_cast<cudaStream_t>(stream)>>>(
      *grid, points, dtype, len, robot_xy, n_frames, pitch, K, stride);
  return check_launch("occ_update_kernel");
}

int b200icp_occ_filter_points(const void* points, int32_t dtype, int32_t cols, int64_t n, const float* probs,
                              int32_t h, int32_t w, double center_x, double center_y, double resolution,
                              float free_threshold, int64_t* kept_index, int64_t* count_out,
                              int64_t* scratch, void* stream) {
  if (!points || !probs || !kept_index || !count_out || !scratch || n < 0 || h < 1 || w < 1 || cols < 2 ||
      !(resolution > 0.0))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "occ_filter_points: bad arguments");
  if (dtype != B200ICP_F32 && dtype != B200ICP_F64) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "occ_filter_points: bad dtype");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (dtype == B200ICP_F64)
    return compact(OccKeep<double>{reinterpret_cast<const double*>(points), cols, probs, h, w, center_x, center_y,
                                   resolution, free_threshold},
                   KeptIndex{kept_index}, n, scratch, count_out, st, "occ_filter");
  return compact(OccKeep<float>{reinterpret_cast<const float*>(points), cols, probs, h, w, center_x, center_y,
                                resolution, free_threshold},
                 KeptIndex{kept_index}, n, scratch, count_out, st, "occ_filter");
}

}  // extern "C"
