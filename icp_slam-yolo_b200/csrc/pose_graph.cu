// pose_graph.cu -- the loop-closure back end: loop-candidate selection from a trajectory, the
// information matrix of an alignment, graph edges from verified alignments and a batched float64
// Gauss-Newton SE(2) pose-graph optimiser whose PCG solve runs on the device (DESIGN.md §4.9).
// The reference has no loop closure: oracle/pose_graph_oracle.py defines the results.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "compact.cuh"
#include "workspace.cuh"

namespace {

constexpr int64_t kPgMaxNodes = 65536;          // per graph
constexpr int64_t kPgMaxEdges = 1 << 20;        // per graph
constexpr int kPgThreads = 512;                 // one CTA per graph
constexpr int kPgWarps = kPgThreads / 32;
constexpr int kSlot = 34;                        // doubles per edge: A'WA 9, A'WB 9, B'WB 9, A'We 3, B'We 3, chi2 1
constexpr int kNodeDoubles = 34;                 // per node: Jacobi inverse 9, diagonal block 9, x, r, z, p, Hp 3 each,
                                                 // held flag 1 (component label during the set-up)

// ------------------------------------------------------------------------------------
// loop candidates: pair q of the (i < j) triangle in PAIR_TRIANGLE order
// ------------------------------------------------------------------------------------
struct CandidateKeep {
  b200icp_problem tri;     // TRIANGLE pairing over the n poses (resolve_rows)
  const double* poses;
  int64_t min_gap;
  double r2;
  __device__ __forceinline__ bool operator()(int64_t q) const {
    int64_t j, i;
    resolve_rows(tri, q, j, i);
    if (j - i < min_gap) return false;
    const double* a = poses + 6 * i;
    const double* b = poses + 6 * j;
    return dist2_f64(a[4], a[5], make_double2(b[4], b[5])) <= r2;
  }
};

struct CandidateEmit {
  b200icp_problem tri;
  const double* poses;
  int64_t capacity;
  int32_t* src_row;
  int32_t* tgt_row;
  double* rel;
  __device__ __forceinline__ void operator()(int64_t dst, int64_t q) const {
    if (dst >= capacity) return;
    int64_t j, i;
    resolve_rows(tri, q, j, i);
    src_row[dst] = (int32_t)j;
    tgt_row[dst] = (int32_t)i;
    // X_i^-1 X_j = (Ri^T Rj, Ri^T (tj - ti)), every product and sum rounded on its own (no FMA)
    const double* a = poses + 6 * i;
    const double* b = poses + 6 * j;
    const double dx = __dsub_rn(b[4], a[4]), dy = __dsub_rn(b[5], a[5]);
    double* o = rel + 6 * dst;
    o[0] = __dadd_rn(__dmul_rn(a[0], b[0]), __dmul_rn(a[2], b[2]));
    o[1] = __dadd_rn(__dmul_rn(a[0], b[1]), __dmul_rn(a[2], b[3]));
    o[2] = __dadd_rn(__dmul_rn(a[1], b[0]), __dmul_rn(a[3], b[2]));
    o[3] = __dadd_rn(__dmul_rn(a[1], b[1]), __dmul_rn(a[3], b[3]));
    o[4] = __dadd_rn(__dmul_rn(a[0], dx), __dmul_rn(a[2], dy));
    o[5] = __dadd_rn(__dmul_rn(a[1], dx), __dmul_rn(a[3], dy));
  }
};

// ------------------------------------------------------------------------------------
// information matrix of an alignment, one warp per pair
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) information_kernel(const b200icp_problem pr, int64_t n_pairs,
                                                          const double* __restrict__ pose,
                                                          const int32_t* __restrict__ indices, double gate,
                                                          int use_gate, double* __restrict__ info,
                                                          int32_t* __restrict__ inliers) {
  const int lane = threadIdx.x & 31;
  const int64_t p = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (p >= n_pairs) return;
  int64_t srow, trow;
  resolve_rows(pr, p, srow, trow);
  int n, m;
  row_lengths(pr, srow, trow, n, m);
  const Se2 P = se2_load(pose + 6 * p);
  const int64_t soff = srow * pr.src_pitch, toff = trow * pr.tgt_pitch;
  // v = (count, sum -q_y, sum q_x, sum q_x^2 + q_y^2)
  double v[4] = {0.0, 0.0, 0.0, 0.0};
  for (int i = lane; i < n; i += 32) {
    const int k = indices[p * pr.src_pitch + i];
    if (k < 0 || k >= m) continue;
    const double2 q = load_point(pr.tgt_points, pr.dtype, toff + k);
    const double2 s = apply(P, load_point(pr.src_points, pr.dtype, soff + i));
    if (use_gate && !(sqrt(dist2_f64(s.x, s.y, q)) < gate)) continue;
    v[0] = __dadd_rn(v[0], 1.0);
    v[1] = __dsub_rn(v[1], q.y);
    v[2] = __dadd_rn(v[2], q.x);
    v[3] = __dadd_rn(v[3], __dadd_rn(__dmul_rn(q.x, q.x), __dmul_rn(q.y, q.y)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int c = 0; c < 4; ++c) v[c] = __dadd_rn(v[c], __shfl_xor_sync(kFull, v[c], o));
  }
  if (lane == 0) {
    double* o = info + 6 * p;
    o[0] = v[0]; o[1] = 0.0; o[2] = v[1]; o[3] = v[0]; o[4] = v[2]; o[5] = v[3];
    if (inliers) inliers[p] = (int32_t)v[0];
  }
}

// ------------------------------------------------------------------------------------
// edges from alignment results
// ------------------------------------------------------------------------------------
struct LoopKeep {
  const double* rmse;
  const int32_t* inliers;
  const int32_t* src_len;
  const int32_t* src_row;
  int32_t src_pitch;
  double min_fitness, max_rmse;
  __device__ __forceinline__ bool operator()(int64_t p) const {
    const double r = rmse[p];
    if (!isfinite(r) || !(r <= max_rmse)) return false;
    const int n = src_len ? min(src_len[src_row[p]], src_pitch) : src_pitch;
    const double fit = n > 0 ? (double)inliers[p] / (double)n : 0.0;
    return fit >= min_fitness;
  }
};

struct OdometryKeep {
  const double* error;
  const int32_t* iterations;
  __device__ __forceinline__ bool operator()(int64_t p) const {
    return iterations[p] > 0 && error[p] != CUDART_INF;
  }
};

struct EdgeEmit {
  const double* pose;
  const double* info;     // NULL: identity information
  const int32_t* src_row; // NULL: odometry, pair p joins (p, p + 1)
  const int32_t* tgt_row;
  int32_t* edge_i;
  int32_t* edge_j;
  double* meas;
  double* info_out;
  __device__ __forceinline__ void operator()(int64_t dst, int64_t p) const {
    edge_i[dst] = src_row ? tgt_row[p] : (int32_t)p;
    edge_j[dst] = src_row ? src_row[p] : (int32_t)(p + 1);
    for (int c = 0; c < 6; ++c) {
      meas[6 * dst + c] = pose[6 * p + c];
      info_out[6 * dst + c] = info ? info[6 * p + c] : (c == 0 || c == 3 || c == 5 ? 1.0 : 0.0);
    }
  }
};

// ------------------------------------------------------------------------------------
// pose-graph optimiser
// ------------------------------------------------------------------------------------
struct PgGraphs {          // device copies of the ragged ranges
  const int64_t* node_offset;
  const int64_t* edge_offset;
  const int32_t* fixed;
};

// key of both slots of every edge: the global node index (graph node offset + local index); a graph
// with an endpoint outside [0, n) or i == j is flagged bad and keys those slots past every node.
__global__ void __launch_bounds__(256) pg_keys_kernel(PgGraphs g, const int32_t* __restrict__ ei,
                                                      const int32_t* __restrict__ ej, int64_t nodes, int32_t* keys,
                                                      int32_t* vals, int32_t* bad) {
  const int64_t gi = blockIdx.x;
  const int64_t nb = g.node_offset[gi], n = g.node_offset[gi + 1] - nb;
  const int64_t eb = g.edge_offset[gi], ne = g.edge_offset[gi + 1] - eb;
  int flag = 0;
  for (int64_t e = eb + threadIdx.x; e < eb + ne; e += blockDim.x) {
    const int32_t a = ei[e], b = ej[e];
    const bool ok = a >= 0 && b >= 0 && a < n && b < n && a != b;
    flag |= !ok;
    keys[2 * e] = (int32_t)(ok ? nb + a : nodes); keys[2 * e + 1] = (int32_t)(ok ? nb + b : nodes);
    vals[2 * e] = (int32_t)e; vals[2 * e + 1] = (int32_t)e;
  }
  flag = __syncthreads_or(flag);
  if (threadIdx.x == 0) bad[gi] = flag;
}

// row_ptr[k] = first slot of node k in the sorted keys (lower bound), row_ptr[nodes] = slots
__global__ void __launch_bounds__(256) pg_rows_kernel(const int32_t* __restrict__ keys, int64_t slots, int64_t nodes,
                                                      int32_t* row_ptr) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k > nodes) return;
  int64_t lo = 0, hi = slots;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < k) lo = mid + 1; else hi = mid;
  }
  row_ptr[k] = (int32_t)lo;
}

// Sum over the CTA in a fixed order: each warp by the xor butterfly, then the warp totals in warp
// order.  `buf` alternates between two halves of the shared scratch so that one __syncthreads
// per reduction suffices.
__device__ __forceinline__ double cta_sum(double v, double* red, int& rb) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  double* buf = red + rb * kPgWarps;
  rb ^= 1;
  if (lane == 0) buf[warp] = v;
  __syncthreads();
  double s = buf[0];
#pragma unroll
  for (int w = 1; w < kPgWarps; ++w) s += buf[w];
  return s;
}

struct PgArgs {
  PgGraphs g;
  const int32_t* ei;
  const int32_t* ej;
  const double* meas;
  const double* info;
  const int32_t* row_ptr;     // [nodes + 1], global slot indices
  const int32_t* slot_edge;   // [2 * edges] edge of each slot, ascending per node
  const int32_t* bad;
  double* edge_ws;            // [edges][kSlot]
  double* node_ws;            // [nodes][kNodeDoubles]
  b200icp_pose_graph_options opt;
  b200icp_pose_graph_outputs out;
};

// e = t2v(Z^-1 (Xi^-1 Xj)) and its Jacobians A = de/dxi, B = de/dxj (Grisetti et al., §IV), then
// the slots of the edge: A'WA, A'WB, B'WB, A'We, B'We (W = the information matrix) and e'We.
__device__ void linearise_edge(const double* Xi, const double* Xj, const double* Z, const double* inf, double* s) {
  const double ri00 = Xi[0], ri01 = Xi[1], ri10 = Xi[2], ri11 = Xi[3];
  const double rz00 = Z[0], rz01 = Z[1], rz10 = Z[2], rz11 = Z[3];
  const double dx = Xj[4] - Xi[4], dy = Xj[5] - Xi[5];
  const double ux = ri00 * dx + ri10 * dy - Z[4], uy = ri01 * dx + ri11 * dy - Z[5];
  const double q00 = ri00 * Xj[0] + ri10 * Xj[2], q10 = ri01 * Xj[0] + ri11 * Xj[2];
  const double m00 = rz00 * q00 + rz10 * q10, m10 = rz01 * q00 + rz11 * q10;
  double eth = atan2(m10, m00);
  if (eth == -CUDART_PI) eth = CUDART_PI;
  const double e[3] = {rz00 * ux + rz10 * uy, rz01 * ux + rz11 * uy, eth};
  const double s00 = rz00 * ri00 + rz10 * ri01, s01 = rz00 * ri10 + rz10 * ri11;
  const double s10 = rz01 * ri00 + rz11 * ri01, s11 = rz01 * ri10 + rz11 * ri11;
  const double w0 = -ri10 * dx + ri00 * dy, w1 = -ri00 * dx - ri10 * dy;
  const double v0 = rz00 * w0 + rz10 * w1, v1 = rz01 * w0 + rz11 * w1;
  const double A[3][3] = {{-s00, -s01, v0}, {-s10, -s11, v1}, {0.0, 0.0, -1.0}};
  const double B[3][3] = {{s00, s01, 0.0}, {s10, s11, 0.0}, {0.0, 0.0, 1.0}};
  const double W[3][3] = {{inf[0], inf[1], inf[2]}, {inf[1], inf[3], inf[4]}, {inf[2], inf[4], inf[5]}};
  double WA[3][3], WB[3][3], We[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    We[r] = W[r][0] * e[0] + W[r][1] * e[1] + W[r][2] * e[2];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      WA[r][c] = W[r][0] * A[0][c] + W[r][1] * A[1][c] + W[r][2] * A[2][c];
      WB[r][c] = W[r][0] * B[0][c] + W[r][1] * B[1][c] + W[r][2] * B[2][c];
    }
  }
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      s[r * 3 + c] = A[0][r] * WA[0][c] + A[1][r] * WA[1][c] + A[2][r] * WA[2][c];
      s[9 + r * 3 + c] = A[0][r] * WB[0][c] + A[1][r] * WB[1][c] + A[2][r] * WB[2][c];
      s[18 + r * 3 + c] = B[0][r] * WB[0][c] + B[1][r] * WB[1][c] + B[2][r] * WB[2][c];
    }
    s[27 + r] = A[0][r] * We[0] + A[1][r] * We[1] + A[2][r] * We[2];
    s[30 + r] = B[0][r] * We[0] + B[1][r] * We[1] + B[2][r] * We[2];
  }
  s[33] = e[0] * We[0] + e[1] * We[1] + e[2] * We[2];
}

// one CTA per graph: the whole Gauss-Newton loop, PCG solves included, on the device
__global__ void __launch_bounds__(kPgThreads) pose_graph_kernel(const PgArgs a) {
  __shared__ double red[2 * kPgWarps];
  const int tid = threadIdx.x;
  const int64_t gi = blockIdx.x;
  const int64_t nb = a.g.node_offset[gi], n = a.g.node_offset[gi + 1] - nb;
  const int64_t eb = a.g.edge_offset[gi], ne = a.g.edge_offset[gi + 1] - eb;
  const int64_t fixed = a.g.fixed ? a.g.fixed[gi] : 0;
  const b200icp_pose_graph_options& op = a.opt;
  double* X = a.out.poses + 6 * nb;
  double* ND = a.node_ws + kNodeDoubles * nb;
  double* ES = a.edge_ws + (int64_t)kSlot * eb;
  const int32_t* ei = a.ei + eb;
  const int32_t* ej = a.ej + eb;
  const int32_t* rp = a.row_ptr;
  int rb = 0;

  int isolated = 0;
  for (int64_t k = tid; k < n; k += kPgThreads) {
    isolated += (rp[nb + k + 1] == rp[nb + k] && k != fixed) ? 1 : 0;
  }
  isolated = (int)cta_sum((double)isolated, red, rb);

  // ---- one held node per connected component: the gauge for its own component, the lowest-index node
  // for every other one, so that H has no null space.  Labels = lowest node index of the component, by
  // min-propagation over the CSR rows with pointer jumping (monotone, so the unsynchronised reads of a
  // sweep are harmless and the fixed point does not depend on the schedule).
  for (int64_t k = tid; k < n; k += kPgThreads) ND[kNodeDoubles * k + 33] = (double)k;
  __syncthreads();
  for (;;) {
    int changed = 0;
    for (int64_t k = tid; k < n; k += kPgThreads) {
      double* lk = ND + kNodeDoubles * k + 33;
      double m = *lk;
      for (int32_t s = rp[nb + k]; s < rp[nb + k + 1]; ++s) {
        const int64_t e = a.slot_edge[s] - eb;
        const int64_t o = ei[e] == k ? ej[e] : ei[e];
        m = fmin(m, ND[kNodeDoubles * o + 33]);
      }
      m = fmin(m, ND[kNodeDoubles * (int64_t)m + 33]);
      if (m < *lk) { *lk = m; changed = 1; }
    }
    if (!__syncthreads_or(changed)) break;
  }
  const double gauge_label = n > 0 ? ND[kNodeDoubles * fixed + 33] : -1.0;
  int anchored = 0;
  for (int64_t k = tid; k < n; k += kPgThreads) {
    const double l = ND[kNodeDoubles * k + 33];
    if (l == (double)k && l != gauge_label && rp[nb + k + 1] > rp[nb + k]) ++anchored;
  }
  __syncthreads();                           // every label is read before the flags overwrite them
  for (int64_t k = tid; k < n; k += kPgThreads) {
    double* lk = ND + kNodeDoubles * k + 33;
    const double l = *lk;
    *lk = (k == fixed || (l == (double)k && l != gauge_label)) ? 1.0 : 0.0;
  }
  anchored = (int)cta_sum((double)anchored, red, rb);   // syncs: the held flags are visible afterwards
  auto held = [&](int64_t k) -> bool { return ND[kNodeDoubles * k + 33] != 0.0; };

  auto linearise = [&]() -> double {
    double c = 0.0;
    for (int64_t e = tid; e < ne; e += kPgThreads) {
      double* s = ES + kSlot * e;
      linearise_edge(X + 6 * ei[e], X + 6 * ej[e], a.meas + 6 * (eb + e), a.info + 6 * (eb + e), s);
      c += s[33];
    }
    return cta_sum(c, red, rb);          // syncs: the slots are visible afterwards
  };

  int status = B200ICP_PG_CONVERGED, iters = 0, pcg_total = 0;
  double chi2_0 = 0.0, chi2 = 0.0;
  if (a.bad[gi]) {
    status = B200ICP_PG_BAD_EDGE;
  } else {
    chi2 = chi2_0 = linearise();
    if (!isfinite(chi2)) status = B200ICP_PG_NON_FINITE;
    bool converged = chi2 == 0.0, pcg_limit = false, breakdown = false;
    while (status == B200ICP_PG_CONVERGED && !converged && iters < op.max_iterations) {
      // ---- assemble the diagonal blocks and gradients (slots in CSR order), Jacobi inverses, PCG start
      double rz = 0.0;
      for (int64_t k = tid; k < n; k += kPgThreads) {
        double D[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};
        const int32_t s0 = rp[nb + k], s1 = rp[nb + k + 1];
        for (int32_t s = s0; s < s1; ++s) {
          const int64_t e = a.slot_edge[s] - eb;
          const double* sl = ES + kSlot * e;
          const bool first = ei[e] == k;
          for (int c = 0; c < 9; ++c) D[c] += sl[(first ? 0 : 18) + c];
          for (int c = 0; c < 3; ++c) g[c] += sl[(first ? 27 : 30) + c];
        }
        if (s1 == s0 || held(k)) {          // eliminated (held) or untouched: identity block, no step
          for (int c = 0; c < 9; ++c) D[c] = (c % 4 == 0) ? 1.0 : 0.0;
          g[0] = g[1] = g[2] = 0.0;
        } else {
          D[0] += op.damping; D[4] += op.damping; D[8] += op.damping;
        }
        // 3x3 inverse by cofactors (D is symmetric positive definite); identity if it is not invertible
        double* nd = ND + kNodeDoubles * k;
        const double c00 = D[4] * D[8] - D[5] * D[7], c01 = D[5] * D[6] - D[3] * D[8], c02 = D[3] * D[7] - D[4] * D[6];
        const double det = D[0] * c00 + D[1] * c01 + D[2] * c02;
        if (det > 0.0 && isfinite(det)) {
          const double id = 1.0 / det;
          nd[0] = c00 * id; nd[1] = (D[2] * D[7] - D[1] * D[8]) * id; nd[2] = (D[1] * D[5] - D[2] * D[4]) * id;
          nd[3] = c01 * id; nd[4] = (D[0] * D[8] - D[2] * D[6]) * id; nd[5] = (D[2] * D[3] - D[0] * D[5]) * id;
          nd[6] = c02 * id; nd[7] = (D[1] * D[6] - D[0] * D[7]) * id; nd[8] = (D[0] * D[4] - D[1] * D[3]) * id;
        } else {
          for (int c = 0; c < 9; ++c) nd[c] = (c % 4 == 0) ? 1.0 : 0.0;
        }
        double *Dn = nd + 9, *x = nd + 18, *r = nd + 21, *z = nd + 24, *p = nd + 27;
        for (int c = 0; c < 9; ++c) Dn[c] = D[c];
        for (int c = 0; c < 3; ++c) { x[c] = 0.0; r[c] = -g[c]; }
        for (int c = 0; c < 3; ++c) z[c] = nd[c * 3] * r[0] + nd[c * 3 + 1] * r[1] + nd[c * 3 + 2] * r[2];
        for (int c = 0; c < 3; ++c) { p[c] = z[c]; rz += r[c] * z[c]; }
      }
      rz = cta_sum(rz, red, rb);
      const double rz0 = rz, stop = op.pcg_tolerance * op.pcg_tolerance * rz0;
      int it = 0;
      for (; it < op.pcg_max_iterations && rz > stop; ++it) {
        // ---- Hp: the assembled diagonal block, then one A'WB slot per incident edge in CSR order
        double pap = 0.0;
        for (int64_t k = tid; k < n; k += kPgThreads) {
          double* nd = ND + kNodeDoubles * k;
          const double* p = nd + 27;
          double y[3] = {0.0, 0.0, 0.0};
          const int32_t s0 = rp[nb + k], s1 = rp[nb + k + 1];
          if (s1 > s0 && !held(k)) {             // eliminated and untouched nodes: (Hp)_k = 0
            const double* D = nd + 9;
            for (int r = 0; r < 3; ++r) y[r] = D[r * 3] * p[0] + D[r * 3 + 1] * p[1] + D[r * 3 + 2] * p[2];
            for (int32_t s = s0; s < s1; ++s) {
              const int64_t e = a.slot_edge[s] - eb;
              const bool first = ei[e] == k;
              const int64_t o = first ? ej[e] : ei[e];
              if (held(o)) continue;
              const double* q = ND + kNodeDoubles * o + 27;
              const double* C = ES + kSlot * e + 9;   // A'WB: rows of node i, columns of node j
              if (first) {
                for (int r = 0; r < 3; ++r) y[r] += C[r * 3] * q[0] + C[r * 3 + 1] * q[1] + C[r * 3 + 2] * q[2];
              } else {
                for (int r = 0; r < 3; ++r) y[r] += C[r] * q[0] + C[3 + r] * q[1] + C[6 + r] * q[2];
              }
            }
            pap += p[0] * y[0] + p[1] * y[1] + p[2] * y[2];
          }
          double* hp = nd + 30;
          hp[0] = y[0]; hp[1] = y[1]; hp[2] = y[2];
        }
        pap = cta_sum(pap, red, rb);
        if (!(pap > 0.0) || !isfinite(pap)) { breakdown = true; break; }
        const double alpha = rz / pap;
        double rzn = 0.0;
        for (int64_t k = tid; k < n; k += kPgThreads) {
          double* nd = ND + kNodeDoubles * k;
          double *x = nd + 18, *r = nd + 21, *z = nd + 24;
          const double *p = nd + 27, *ap = nd + 30;
          for (int c = 0; c < 3; ++c) { x[c] += alpha * p[c]; r[c] -= alpha * ap[c]; }
          for (int c = 0; c < 3; ++c) z[c] = nd[c * 3] * r[0] + nd[c * 3 + 1] * r[1] + nd[c * 3 + 2] * r[2];
          rzn += r[0] * z[0] + r[1] * z[1] + r[2] * z[2];
        }
        rzn = cta_sum(rzn, red, rb);
        const double beta = rzn / rz;
        rz = rzn;
        for (int64_t k = tid; k < n; k += kPgThreads) {
          double* nd = ND + kNodeDoubles * k;
          for (int c = 0; c < 3; ++c) nd[27 + c] = nd[24 + c] + beta * nd[27 + c];
        }
        __syncthreads();                         // p of every node before the next product
      }
      pcg_total += it;
      if (breakdown) { status = B200ICP_PG_PCG_BREAKDOWN; break; }   // p'Hp not positive: no step applied
      if (rz > stop) pcg_limit = true;
      // ---- X_k <- X_k (+) x_k: t + dt, R R(dtheta)
      int finite_step = 1;
      for (int64_t k = tid; k < n; k += kPgThreads) {
        const double* x = ND + kNodeDoubles * k + 18;
        finite_step &= isfinite(x[0]) && isfinite(x[1]) && isfinite(x[2]);
      }
      if (!__syncthreads_and(finite_step)) { status = B200ICP_PG_NON_FINITE; break; }
      for (int64_t k = tid; k < n; k += kPgThreads) {
        const double* x = ND + kNodeDoubles * k + 18;
        if (x[0] == 0.0 && x[1] == 0.0 && x[2] == 0.0) continue;
        double* P = X + 6 * k;
        double sn, cs;
        sincos(x[2], &sn, &cs);
        const double r00 = P[0], r01 = P[1], r10 = P[2], r11 = P[3];
        P[0] = r00 * cs + r01 * sn; P[1] = r01 * cs - r00 * sn;
        P[2] = r10 * cs + r11 * sn; P[3] = r11 * cs - r10 * sn;
        P[4] += x[0]; P[5] += x[1];
      }
      ++iters;
      __syncthreads();                           // poses before the next linearisation
      const double c = linearise();
      if (!isfinite(c)) { chi2 = c; status = B200ICP_PG_NON_FINITE; break; }
      converged = fabs(chi2 - c) <= op.tolerance * chi2 || c == 0.0;
      chi2 = c;
    }
    if (status == B200ICP_PG_CONVERGED) {
      if (pcg_limit) status = B200ICP_PG_PCG_LIMIT;
      else if (!converged) status = B200ICP_PG_MAX_ITERATIONS;
    }
  }
  if (tid == 0) {
    const b200icp_pose_graph_outputs& o = a.out;
    if (o.chi2_initial) o.chi2_initial[gi] = chi2_0;
    if (o.chi2_final) o.chi2_final[gi] = chi2;
    if (o.iterations) o.iterations[gi] = iters;
    if (o.pcg_iterations) o.pcg_iterations[gi] = pcg_total;
    if (o.isolated) o.isolated[gi] = isolated;
    if (o.anchored) o.anchored[gi] = anchored;
    o.status[gi] = status;
  }
}

struct PgBuffers {
  void* ranges;             // node_offset[G + 1], edge_offset[G + 1] (int64), fixed[G] (int32): one copy
  int32_t *keys, *vals;     // [2 * edges] node and edge of every edge slot
  int32_t *skeys, *svals;   // the same, sorted by node
  int32_t *rows, *bad;      // [nodes + 1], [G]
  double *edge_ws, *node_ws;
  SortTemp sort;
  int64_t bytes;
};

PgBuffers pg_buffers(void* base, int64_t n_graphs, int64_t nodes, int64_t edges) {
  Carver c(base);
  PgBuffers b;
  b.ranges = c.take_bytes(sizeof(int64_t) * 2 * (n_graphs + 1) + sizeof(int32_t) * n_graphs);
  b.keys = c.take<int32_t>(2 * edges);
  b.vals = c.take<int32_t>(2 * edges);
  b.skeys = c.take<int32_t>(2 * edges);
  b.svals = c.take<int32_t>(2 * edges);
  b.rows = c.take<int32_t>(nodes + 1);
  b.bad = c.take<int32_t>(n_graphs);
  b.edge_ws = c.take<double>(kSlot * edges);
  b.node_ws = c.take<double>(kNodeDoubles * nodes);
  b.sort = take_sort_temp<int32_t, int32_t>(c, 2 * edges);
  b.bytes = c.total;
  return b;
}

int pg_sizes(const b200icp_pose_graph_batch* g, int64_t& nodes, int64_t& edges) {
  if (!g || g->n_graphs < 0) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: batch is NULL or n_graphs < 0");
  if (g->n_graphs > 0 && (!g->node_offset || !g->edge_offset))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: node_offset / edge_offset is NULL");
  if (g->n_graphs > 0 && (g->node_offset[0] != 0 || g->edge_offset[0] != 0))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: node_offset[0] and edge_offset[0] must be 0");
  for (int32_t k = 0; k < g->n_graphs; ++k) {
    const int64_t n = g->node_offset[k + 1] - g->node_offset[k], e = g->edge_offset[k + 1] - g->edge_offset[k];
    if (n < 0 || e < 0) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: offsets of graph %d decrease", k);
    if (n > kPgMaxNodes || e > kPgMaxEdges)
      return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "pose_graph: graph %d has %lld nodes / %lld edges (limits 65536 / 2^20)",
                       k, (long long)n, (long long)e);
    const int32_t f = g->fixed_node ? g->fixed_node[k] : 0;
    if (f < 0 || (n > 0 && f >= n))
      return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: fixed node %d of graph %d is outside [0, %lld)", f, k,
                       (long long)n);
  }
  nodes = g->n_graphs > 0 ? g->node_offset[g->n_graphs] : 0;
  edges = g->n_graphs > 0 ? g->edge_offset[g->n_graphs] : 0;
  if (nodes >= (1LL << 31) - 1 || 2 * edges >= (1LL << 31) - 1)
    return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "pose_graph: more than 2^31 nodes or 2^30 edges in one call");
  return B200ICP_OK;
}

}  // namespace

extern "C" {

int b200icp_loop_candidates(const double* poses, int64_t n, int64_t min_gap, double radius, int64_t capacity,
                            int32_t* src_row, int32_t* tgt_row, double* rel_pose, int64_t* count_out,
                            int64_t* scratch, void* stream) {
  if (n < 0 || capacity < 0 || (n > 1 && !poses) || !count_out || !scratch ||
      (capacity > 0 && (!src_row || !tgt_row || !rel_pose)))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "loop_candidates: bad arguments");
  if (min_gap < 1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "loop_candidates: min_gap must be >= 1");
  if (!(radius >= 0.0) || std::isnan(radius)) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "loop_candidates: radius must be >= 0");
  if (n > kPgMaxNodes) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "loop_candidates: more than 65536 poses");
  b200icp_problem tri;
  memset(&tri, 0, sizeof(tri));
  tri.pairing = B200ICP_PAIR_TRIANGLE;
  tri.n_rows = (int32_t)n;
  const double r2 = radius * radius;
  const int64_t pairs = n * (n - 1) / 2;
  return compact(CandidateKeep{tri, poses, min_gap, r2}, CandidateEmit{tri, poses, capacity, src_row, tgt_row, rel_pose},
                 pairs, scratch, count_out, reinterpret_cast<cudaStream_t>(stream), "loop_candidates");
}

int b200icp_information_batch(const b200icp_problem* prob, int64_t n_pairs, const double* pose,
                              const int32_t* indices, double max_corr_dist, double* info_out, int32_t* inliers_out,
                              void* stream) {
  if (const int rc = check_problem(prob, n_pairs, false)) return rc;   // no shared-memory tile: any pitch
  if (!pose || !indices || !info_out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "information_batch: pose / indices / info_out is NULL");
  if (n_pairs == 0) return B200ICP_OK;
  const int use_gate = (max_corr_dist > 0.0 && std::isfinite(max_corr_dist)) ? 1 : 0;
  const int64_t blocks = (n_pairs + 7) / 8;
  if (blocks > 0x7fffffffLL) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "information_batch: too many pairs");
  information_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      *prob, n_pairs, pose, indices, max_corr_dist, use_gate, info_out, inliers_out);
  return check_launch("information_kernel");
}

int b200icp_loop_edges(int64_t n_pairs, const double* pose_total, const double* rmse, const int32_t* inliers,
                       const int32_t* src_len, int32_t src_pitch, const int32_t* src_row, const int32_t* tgt_row,
                       const double* info, double min_fitness, double max_rmse, int32_t* edge_i, int32_t* edge_j,
                       double* meas, double* info_out, int64_t* count_out, int64_t* scratch, void* stream) {
  if (n_pairs < 0 || !count_out || !scratch || src_pitch < 1 ||
      (n_pairs > 0 && (!pose_total || !rmse || !inliers || !src_row || !tgt_row || !edge_i || !edge_j || !meas || !info_out)))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "loop_edges: bad arguments");
  if (std::isnan(min_fitness) || std::isnan(max_rmse)) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "loop_edges: NaN threshold");
  return compact(LoopKeep{rmse, inliers, src_len, src_row, src_pitch, min_fitness, max_rmse},
                 EdgeEmit{pose_total, info, src_row, tgt_row, edge_i, edge_j, meas, info_out}, n_pairs, scratch,
                 count_out, reinterpret_cast<cudaStream_t>(stream), "loop_edges");
}

int b200icp_odometry_edges(int64_t n_pairs, const double* pose_total, const double* error, const int32_t* iterations,
                           const double* info, int32_t* edge_i, int32_t* edge_j, double* meas, double* info_out,
                           int64_t* count_out, int64_t* scratch, void* stream) {
  if (n_pairs < 0 || !count_out || !scratch ||
      (n_pairs > 0 && (!pose_total || !error || !iterations || !edge_i || !edge_j || !meas || !info_out)))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "odometry_edges: bad arguments");
  if (n_pairs >= (1LL << 31) - 1) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "odometry_edges: too many pairs");
  return compact(OdometryKeep{error, iterations},
                 EdgeEmit{pose_total, info, nullptr, nullptr, edge_i, edge_j, meas, info_out}, n_pairs, scratch,
                 count_out, reinterpret_cast<cudaStream_t>(stream), "odometry_edges");
}

int64_t b200icp_pose_graph_workspace_bytes(const b200icp_pose_graph_batch* graphs) {
  int64_t nodes = 0, edges = 0;
  if (pg_sizes(graphs, nodes, edges) != B200ICP_OK) return -1;
  return pg_buffers(nullptr, graphs->n_graphs, nodes, edges).bytes;
}

int b200icp_pose_graph_optimize(const b200icp_pose_graph_batch* graphs, const b200icp_pose_graph_options* opt,
                                const b200icp_pose_graph_outputs* out, void* workspace, int64_t workspace_bytes,
                                void* stream) {
  int64_t nodes = 0, edges = 0;
  if (const int rc = pg_sizes(graphs, nodes, edges)) return rc;
  if (!opt || !out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: options / outputs is NULL");
  if (opt->max_iterations < 0 || opt->pcg_max_iterations < 0 || !(opt->tolerance >= 0.0) ||
      !(opt->pcg_tolerance >= 0.0) || !(opt->damping >= 0.0) || !std::isfinite(opt->damping))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: negative / NaN option");
  if (graphs->n_graphs > 0 && !out->status) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: outputs.status is required");
  if (nodes > 0 && (!graphs->poses_in || !out->poses))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: poses_in / outputs.poses is NULL");
  if (edges > 0 && (!graphs->edge_i || !graphs->edge_j || !graphs->meas || !graphs->info))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: edge arrays are NULL");
  if (graphs->n_graphs == 0) return B200ICP_OK;
  const int64_t G = graphs->n_graphs;
  const PgBuffers b = pg_buffers(workspace, G, nodes, edges);
  if (!workspace || workspace_bytes < b.bytes)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_graph: workspace smaller than b200icp_pose_graph_workspace_bytes()");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // the ranges and the gauge nodes travel to the device once per call
  std::vector<char> host(sizeof(int64_t) * 2 * (G + 1) + sizeof(int32_t) * G);
  memcpy(host.data(), graphs->node_offset, sizeof(int64_t) * (G + 1));
  memcpy(host.data() + sizeof(int64_t) * (G + 1), graphs->edge_offset, sizeof(int64_t) * (G + 1));
  int32_t* hf = reinterpret_cast<int32_t*>(host.data() + sizeof(int64_t) * 2 * (G + 1));
  for (int64_t k = 0; k < G; ++k) hf[k] = graphs->fixed_node ? graphs->fixed_node[k] : 0;
  cudaError_t e = cudaMemcpyAsync(b.ranges, host.data(), host.size(), cudaMemcpyHostToDevice, st);
  // (a copy from pageable memory is staged before cudaMemcpyAsync returns, so `host` may go out of scope)
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "pose_graph: ranges to the device: %s", cudaGetErrorString(e));
  PgGraphs pg;
  pg.node_offset = static_cast<const int64_t*>(b.ranges);
  pg.edge_offset = pg.node_offset + (G + 1);
  pg.fixed = reinterpret_cast<const int32_t*>(pg.edge_offset + (G + 1));
  // ---- set-up: block-CSR of H (each node's slots in ascending edge order: the sort is stable)
  pg_keys_kernel<<<(unsigned)G, 256, 0, st>>>(pg, graphs->edge_i, graphs->edge_j, nodes, b.keys, b.vals, b.bad);
  if (const int rc = check_launch("pg_keys_kernel")) return rc;
  if (edges > 0) {
    int bits = 1;
    while (bits < 31 && (1LL << bits) <= nodes) ++bits;
    if (const int rc = radix_sort_pairs(b.sort, b.keys, b.skeys, b.vals, b.svals, 2 * edges, 0, bits, st,
                                        "pose_graph: radix sort"))
      return rc;
  }
  pg_rows_kernel<<<(unsigned)((nodes + 256) / 256), 256, 0, st>>>(b.skeys, 2 * edges, nodes, b.rows);
  if (const int rc = check_launch("pg_rows_kernel")) return rc;
  if (nodes > 0) {
    e = cudaMemcpyAsync(out->poses, graphs->poses_in, sizeof(double) * 6 * nodes, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "pose_graph: pose copy: %s", cudaGetErrorString(e));
  }
  PgArgs args;
  args.g = pg;
  args.ei = graphs->edge_i;
  args.ej = graphs->edge_j;
  args.meas = graphs->meas;
  args.info = graphs->info;
  args.row_ptr = b.rows;
  args.slot_edge = b.svals;
  args.bad = b.bad;
  args.edge_ws = b.edge_ws;
  args.node_ws = b.node_ws;
  args.opt = *opt;
  args.out = *out;
  pose_graph_kernel<<<(unsigned)G, kPgThreads, 0, st>>>(args);
  return check_launch("pose_graph_kernel");
}

}  // extern "C"
