// Solve routines of the B200 ESIKF update: the Kalman gain, the boxplus state update, loop control and the final
// covariance update. The whole iteration loop runs on the device with no host round trip.
//
//   lio_solve_block / lio_solve_kernel : src/voxel_map.cpp:462-499  (K_1, G, solution, state_ += solution, convergence /
//                                        rematch / (I-G)P)
//   vio_solve_block / vio_solve_kernel : src/vio.cpp:1636-1685 + :800 (error-gated accept / rollback, K_1, G, solution, final
//                                        cov -= G cov)
//
// Gain: the reference computes K_1 = (H^T H + P^-1)^-1 with two 19x19 partial-pivot inversions and then only uses the
// first m (6 or 7) columns of K_1. Because H^T H is zero outside its leading m x m block A, the push-through identity gives
//     K_1[:, :m] = P[:, :m] (I_m + A P_mm)^-1
// exactly — an m x m solve with 19 right-hand sides, one per lane. solve_mode 1 keeps the literal double inversion (Gauss-
// Jordan with partial pivoting in shared memory) for parity checks.
//
// Critical path inside the persistent kernels: [all CTAs arrived] -> sum of the partial columns -> gain elimination ->
// boxplus -> next slice. Everything that does not need the new information vector is hoisted out of it:
// state_propagat (-) state is evaluated by warp 1 while the CTA waits at the grid barrier, and P never changes inside the
// loop. The elimination itself is one warp, one column per lane.
#include <float.h>
#include "esikf_dev.cuh"

namespace esikf {

struct SolveArgs {
  double *state;        // current iterate (device, packed) — updated in place
  const double *prop;   // state_propagat
  const double *info;   // reduced information vector (compact, NE_MAX doubles)
  Ctrl *ctrl;
  int max_iterations;
  int solve_mode;
  // LIO
  esikf_lio_stats *lio_stats;
  // VIO
  esikf_vio_stats *vio_stats;
  double *old_state;    // 25 doubles (pose part of old_state)
  double *G;            // 19 x 7 last accepted gain block
  double img_point_cov;
  int level, slot_iter, last_slot;
  int no_publish;       // persistent kernels: every CTA solves, only one CTA writes the results to global memory
  unsigned long long *dbg;  // measurement only: [0] gain rows done, [1] boxplus done (thread 0)
};

struct SolveSmem {
  double P[19 * 19];
  double A[49];     // m x m information block (full, mirrored from the upper triangle)
  double HTz[8];
  double vec[19];
  double sol[19];
  double *W;        // literal mode (solve_mode 1) workspace, 19 x 38 doubles
  double *K;        // literal mode, 19 x 19 doubles
  // loop invariants of the gain (P does not change inside an update), gain_setup:
  double Sinv[49];  // (P_mm pscale)^-1, m x m
  double B[19][8];  // P[:, :m] P_mm^-1, 19 x m
};
struct SolveLiteralScratch {
  double W[19 * 38];
  double K[19 * 19];
};

// Exp(v) of include/utils/so3_math.h:44-58 (identity when |v| <= 1e-5)
__device__ inline void so3_exp(const double v[3], double E[9]) {
  double nrm = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  for (int i = 0; i < 9; i++) E[i] = (i % 4 == 0) ? 1.0 : 0.0;
  if (nrm > 0.00001) {
    double r[3] = {v[0] / nrm, v[1] / nrm, v[2] / nrm};
    double K[9] = {0.0, -r[2], r[1], r[2], 0.0, -r[0], -r[1], r[0], 0.0};
    double s, cc;
    sincos(nrm, &s, &cc);
    const double c = 1.0 - cc;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) {
        double kk = K[i * 3] * K[j] + K[i * 3 + 1] * K[3 + j] + K[i * 3 + 2] * K[6 + j];
        E[i * 3 + j] = E[i * 3 + j] + s * K[i * 3 + j] + c * kk;
      }
  }
}
// Log(R) of include/utils/so3_math.h:61-66
__device__ inline void so3_log(const double R[9], double out[3]) {
  double tr = R[0] + R[4] + R[8];
  double theta = (tr > 3.0 - 1e-6) ? 0.0 : acos(0.5 * (tr - 1));
  double K[3] = {R[7] - R[5], R[2] - R[6], R[3] - R[1]};
  double f = (fabs(theta) < 0.001) ? 0.5 : (0.5 * theta / sin(theta));
  for (int i = 0; i < 3; i++) out[i] = f * K[i];
}

// packed offsets of the additive blocks in error-state order: p(3:6) expo(6) v(7:10) bg(10:13) ba(13:16) g(16:19)
__device__ __forceinline__ int err_to_packed(int k) {
  return (k < 6) ? S_P + (k - 3) : (k == 6) ? S_EXPO : (k < 10) ? S_V + (k - 7) : (k < 13) ? S_BG + (k - 10) : (k < 16) ? S_BA + (k - 13) : S_G + (k - 16);
}

// vec = state_propagat (-) state  (common_lib.h:194-206), by one warp (lane 0 does the rotation part)
__device__ inline void boxminus_warp(const double *prop, const double *st, double *vec, int lane) {
  if (lane == 0) {
    double Rd[9];
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) Rd[i * 3 + j] = st[S_R + 0 * 3 + i] * prop[S_R + 0 * 3 + j] + st[S_R + 1 * 3 + i] * prop[S_R + 1 * 3 + j] +
                                                   st[S_R + 2 * 3 + i] * prop[S_R + 2 * 3 + j];  // b.rot^T * this.rot
    double l[3];
    so3_log(Rd, l);
    vec[0] = l[0], vec[1] = l[1], vec[2] = l[2];
  }
  if (lane >= 3 && lane < 19) {
    const int off = err_to_packed(lane);
    vec[lane] = prop[off] - st[off];
  }
}

// state (+)= sol  (common_lib.h:182-192) by one warp: every lane evaluates Exp (same instructions, no divergence cost),
// lanes 0..8 each form one entry of R * Exp(sol[0:3]), lanes 3..18 add the vector blocks.
__device__ inline void boxplus_warp(double *st, const double *sol, int lane) {
  double E[9];
  so3_exp(sol, E);
  double rn = 0.0;
  if (lane < 9) {
    const int i = lane / 3, j = lane - 3 * i;
    rn = st[S_R + i * 3] * E[j] + st[S_R + i * 3 + 1] * E[3 + j] + st[S_R + i * 3 + 2] * E[6 + j];
  }
  __syncwarp();
  if (lane < 9) st[S_R + lane] = rn;
  if (lane >= 3 && lane < 19) st[err_to_packed(lane)] += sol[lane];
}

// In-place inverse of a 19x19 in shared memory by one warp (Gauss-Jordan, partial pivoting) — literal mode only.
__device__ inline void inverse19_warp(const double *Ain, double *W /*19x38*/, double *out, int lane) {
  for (int idx = lane; idx < 19 * 38; idx += 32) {
    int r = idx / 38, c = idx % 38;
    W[idx] = (c < 19) ? Ain[r * 19 + c] : ((c - 19) == r ? 1.0 : 0.0);
  }
  __syncwarp();
  for (int k = 0; k < 19; k++) {
    int piv = k;
    double best = fabs(W[k * 38 + k]);
    for (int r = k + 1; r < 19; r++) {
      double v = fabs(W[r * 38 + k]);
      if (v > best) best = v, piv = r;
    }
    __syncwarp();
    if (piv != k)
      for (int c = lane; c < 38; c += 32) {
        double t = W[k * 38 + c];
        W[k * 38 + c] = W[piv * 38 + c];
        W[piv * 38 + c] = t;
      }
    __syncwarp();
    double d = W[k * 38 + k];
    double f[19];
    for (int r = 0; r < 19; r++) f[r] = W[r * 38 + k];
    __syncwarp();
    for (int c = lane; c < 38; c += 32) {
      double pk = W[k * 38 + c] / d;
      W[k * 38 + c] = pk;
      for (int r = 0; r < 19; r++)
        if (r != k) W[r * 38 + c] -= f[r] * pk;
    }
    __syncwarp();
  }
  for (int idx = lane; idx < 361; idx += 32) out[idx] = W[(idx / 19) * 38 + 19 + (idx % 19)];
  __syncwarp();
}

// Gain. With S = P_mm pscale (pscale = 1 for LIO, 1/img_point_cov for VIO) and A = H^T R^-1 H:
//     K_1[:, :m] = P[:, :m] pscale (I + A S)^-1 = (P[:, :m] P_mm^-1) (S^-1 + A)^-1 = B C^-1,
// where B (19 x m) and S^-1 only depend on P — loop invariants, formed once per update by gain_setup — and C = S^-1 + A is
// symmetric positive definite, so the per-iteration elimination needs no pivot search and no row exchanges: m steps of
// {broadcast the pivot column, reciprocal, rank-1 update}, one column per lane. That is what sits on the critical path of
// every iteration (all CTAs wait for it), and it is a third of the instructions of the pivoted elimination on I + A S.
//
// One elimination sweep of the augmented system [C | RHS columns], one column per lane (col[i] = entry in row i), without
// pivoting: afterwards a right-hand-side lane holds its solution vector.
template <int m> __device__ __forceinline__ void spd_sweep(double col[m]) {
#pragma unroll
  for (int k = 0; k < m; k++) {
    const double pv = __shfl_sync(0xffffffffu, col[k], k);
    double f[m];
#pragma unroll
    for (int i = 0; i < m; i++) f[i] = __shfl_sync(0xffffffffu, col[i], k);
    const double vk = col[k] * __drcp_rn(pv);  // correctly rounded reciprocal: the value of 1.0 / pv without the division subroutine
    col[k] = vk;
#pragma unroll
    for (int i = 0; i < m; i++)
      if (i != k) col[i] -= f[i] * vk;
  }
}

// Once per update, by one warp: S^-1 and B = P[:, :m] P_mm^-1 into shared memory. Lanes 0..m-1 own the columns of S (SPD),
// lanes m..18 the right-hand sides P[r, :m] pscale (rows r >= m of B; rows r < m are unit vectors), lanes 19..19+m-1 the
// unit vectors (rows of S^-1): 19 + m <= 26 columns.
template <int m> __device__ inline void gain_setup(SolveSmem &sm, double pscale, int lane) {
  double col[m];
#pragma unroll
  for (int i = 0; i < m; i++) {
    double v = 0.0;
    if (lane < 19) v = sm.P[lane * 19 + i] * pscale;  // column `lane` of S for lane < m (S symmetric), row `lane` of P[:, :m] otherwise
    else if (lane < 19 + m) v = (i == lane - 19) ? 1.0 : 0.0;
    col[i] = v;
  }
  spd_sweep<m>(col);
#pragma unroll
  for (int i = 0; i < m; i++) {
    if (lane < m) sm.B[lane][i] = (i == lane) ? 1.0 : 0.0;
    else if (lane < 19) sm.B[lane][i] = col[i];
    else if (lane < 19 + m) sm.Sinv[(lane - 19) * m + i] = col[i];
  }
  __syncwarp();
}

// Gain block x = K_1[lane, 0:m] for every lane < 19 (needs gain_setup<m> on this sm for solve_mode 0).
template <int m>
__device__ inline void gain_rows(SolveSmem &sm, double pscale, int solve_mode, int lane, double x[m]) {
  if (solve_mode == 1) {
    // literal: K_1 = (H_T_H + (P*pscale)^-1)^-1
    for (int idx = lane; idx < 361; idx += 32) sm.K[idx] = sm.P[idx] * pscale;
    __syncwarp();
    inverse19_warp(sm.K, sm.W, sm.K, lane);
    for (int idx = lane; idx < m * m; idx += 32) sm.K[(idx / m) * 19 + (idx % m)] += sm.A[idx];
    __syncwarp();
    inverse19_warp(sm.K, sm.W, sm.K, lane);
    if (lane < 19)
      for (int j = 0; j < m; j++) x[j] = sm.K[lane * 19 + j];
    return;
  }
  // lane c < m: column c of C = S^-1 + A (symmetric); lane m + r: right-hand side B[r, :] of state row r
  double col[m];
  if (lane < m) {
#pragma unroll
    for (int i = 0; i < m; i++) col[i] = sm.Sinv[i * m + lane] + sm.A[i * m + lane];
  } else {
    const int r = (lane - m) < 19 ? (lane - m) : 0;
#pragma unroll
    for (int i = 0; i < m; i++) col[i] = sm.B[r][i];
  }
  spd_sweep<m>(col);
#pragma unroll
  for (int i = 0; i < m; i++) x[i] = __shfl_sync(0xffffffffu, col[i], (lane + m) & 31);
}

__device__ inline double warp_norm3(const double *v) { return sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }

#define SOLVE_THREADS 512

// Staging shared by both solve routines: one global round trip brings P, info, the pose parts of state / prior / old_state.
struct SolveIO {
  double info[NE_MAX];
  double st[32];   // first 25 doubles of the packed state (R p expo v bg ba g)
  double pr[32];   // same of state_propagat
  double old[32];  // VIO old_state
  double g[19][8]; // gain block G[:, :m]
  int flags[8];
};

// Needs >= 192 threads. Every global load is issued before the first shared-memory store, so the staging costs one
// L2 round trip.
__device__ __forceinline__ void solve_load(SolveSmem &sm, SolveIO &io, const SolveArgs &a, bool want_old) {
  const int t = threadIdx.x, nt = blockDim.x;
  const double p0 = (t < 361) ? __ldcg(a.state + S_COV + t) : 0.0;
  const double p1 = (t + nt < 361) ? __ldcg(a.state + S_COV + t + nt) : 0.0;
  const double i0 = (t < NE_MAX) ? __ldcg(a.info + t) : 0.0;
  const double s0 = (t < 25) ? __ldcg(a.state + t) : 0.0;
  const double r0 = (t < 25) ? a.prop[t] : 0.0;
  const double o0 = (want_old && t < 25) ? __ldcg(a.old_state + t) : 0.0;
  if (t < 361) sm.P[t] = p0;
  if (t + nt < 361) sm.P[t + nt] = p1;
  if (t < NE_MAX) io.info[t] = i0;
  if (t < 25) {
    io.st[t] = s0;
    io.pr[t] = r0;
    if (want_old) io.old[t] = o0;
  }
}

// m x m information block and H^T z out of the compact vector (mirrored), by one warp.
template <int M> __device__ __forceinline__ void unpack_info(SolveSmem &sm, const SolveIO &io, int lane) {
  constexpr int T = M * (M + 1) / 2;
  for (int idx = lane; idx < M * M; idx += 32) {
    const int i = idx / M, j = idx - M * i;
    sm.A[idx] = io.info[(i <= j) ? tri_of(M, i, j) : tri_of(M, j, i)];
  }
  if (lane < M) sm.HTz[lane] = io.info[T + lane];
  __syncwarp();
}
#define INFO_EXTRA(M) ((M) * ((M) + 1) / 2 + (M))      // sum |d| / sum res^2
#define INFO_COUNTM(M) ((M) * ((M) + 1) / 2 + (M) + 1) // matched points / n_meas

// Diagnostics of the iteration just solved (what the reference prints at voxel_map.cpp:404-405): plain global stores by a
// few threads, nobody inside the kernel reads them.
__device__ __forceinline__ void lio_write_stats(const SolveArgs &a, SolveSmem &sm, SolveIO &io) {
  const int tid = threadIdx.x, iterCount = io.flags[3];
  if (a.lio_stats && iterCount < 8) {
    esikf_lio_stats &S = *a.lio_stats;
    for (int t = tid; t < 36; t += blockDim.x) S.HTH[iterCount][t] = sm.A[t];
    for (int t = tid; t < 6; t += blockDim.x) S.HTz[iterCount][t] = sm.HTz[t];
    for (int t = tid; t < 19; t += blockDim.x) S.solution[iterCount][t] = sm.sol[t];
    if (tid == 0) {
      S.iters = iterCount + 1;
      S.effct_feat_num[iterCount] = (int)io.info[INFO_COUNTM(6)];
      S.total_residual[iterCount] = io.info[INFO_EXTRA(6)];
      S.converged[iterCount] = io.flags[0];
    }
  }
}

// One LIO gain solve + state update (src/voxel_map.cpp:462-499) by the calling block. Returns EKF_stop_flg.
// `ctrl` is the loop-control block the routine reads and updates (the CTA's shared-memory copy). P, the poses and info are
// staged in sm / io, state_propagat (-) state_ is in sm.vec (:470) and, in solve mode 0, gain_setup<6> has run.
__device__ __noinline__ bool lio_solve_block(const SolveArgs &a, SolveSmem &sm, SolveIO &io, Ctrl &ctrl) {
  const int tid = threadIdx.x, lane = tid & 31;
  const int iterCount = ctrl.iter;
  const int rematch0 = ctrl.rematch_num;
  if (tid < 32) {
    unpack_info<6>(sm, io, lane);  // H^T R^-1 H, H^T R^-1 z
    double x[6], g[6];
    gain_rows<6>(sm, 1.0, a.solve_mode, lane, x);
    if (a.dbg && tid == 0) a.dbg[0] = globaltimer_ns();
    // G[lane, 0:6] = K_1[lane, 0:6] * HTH   (voxel_map.cpp:469)
#pragma unroll
    for (int j = 0; j < 6; j++) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) s += x[k] * sm.A[k * 6 + j];
      g[j] = s;
    }
    // solution = K_1[:, :6] HTz + vec - G[:, :6] vec[:6]   (:471-472)
    if (lane < 19) {
      double s1 = 0.0, s2 = 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) s1 += x[k] * sm.HTz[k], s2 += g[k] * sm.vec[k];
      sm.sol[lane] = s1 + sm.vec[lane] - s2;
#pragma unroll
      for (int j = 0; j < 6; j++) io.g[lane][j] = g[j];
    }
    __syncwarp();
    boxplus_warp(io.st, sm.sol, lane);  // state_ += solution (:474)
    if (a.dbg && tid == 0) a.dbg[1] = globaltimer_ns();
    if (lane == 0) {
      const bool converged = (warp_norm3(sm.sol) * 57.3 < 0.01) && (warp_norm3(sm.sol + 3) * 100 < 0.015);  // :477
      int rematch = rematch0;
      if (converged || ((rematch == 0) && (iterCount == (a.max_iterations - 2)))) rematch++;  // :482
      const bool stop = (rematch >= 2) || (iterCount == a.max_iterations - 1);                // :485
      io.flags[0] = converged, io.flags[1] = rematch, io.flags[2] = stop, io.flags[3] = iterCount;
      ctrl.iter = iterCount + 1;
      ctrl.rematch_num = rematch;
      ctrl.stop = stop ? 1 : 0;
    }
  }
  __syncthreads();
  const bool stop = io.flags[2] != 0;
  if (!a.no_publish) {
    for (int t = tid; t < 25; t += blockDim.x) a.state[t] = io.st[t];
    if (stop) {
      // cov = (I - G) cov   (:489-490); G only has its first 6 columns
      for (int t = tid; t < 361; t += blockDim.x) {
        const int r = t / 19, c = t - 19 * r;
        double s = sm.P[t];
#pragma unroll
        for (int j = 0; j < 6; j++) s -= io.g[r][j] * sm.P[j * 19 + c];
        a.state[S_COV + t] = s;
      }
    }
    lio_write_stats(a, sm, io);
  }
  return stop;
}

// Shared memory of the stand-alone solve kernels (one launch per iteration, nothing kept between launches).
struct SolveKernelSmem {
  SolveSmem sm;
  SolveIO io;
  SolveLiteralScratch lit;
  Ctrl ctrl;
};

// Prologue of the stand-alone solve kernels (m = 6: LIO, 7: VIO): the loop control and what the persistent kernels keep
// resident — P, the poses and info, vec = state_propagat (-) state and, in solve mode 0, the gain invariants. A VIO level
// that already ended (EKF_end, vio.cpp:1685) runs no solve, and on its last slot only the final covariance pass, which
// needs neither vec nor the gain. Returns whether the solve routine runs.
template <int m> __device__ __forceinline__ bool solve_kernel_prologue(const SolveArgs &a, SolveKernelSmem &s, double pscale) {
  constexpr bool vio = (m == 7);
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid == 0) s.sm.W = s.lit.W, s.sm.K = s.lit.K, s.ctrl = *a.ctrl;
  __syncthreads();
  const bool level_done = vio && a.slot_iter != 0 && s.ctrl.level_done;  // entering a level: EKF_end = false (vio.cpp:1527)
  if (level_done && !a.last_slot) return false;
  solve_load(s.sm, s.io, a, vio && a.slot_iter != 0);
  __syncthreads();
  if (!level_done) {
    if (tid >= 32 && tid < 64) boxminus_warp(s.io.pr, s.io.st, s.sm.vec, lane);
    if (tid >= 64 && tid < 96 && a.solve_mode == 0) gain_setup<m>(s.sm, pscale, lane);
    __syncthreads();
  }
  return true;
}

__global__ void __launch_bounds__(SOLVE_THREADS, 1) lio_solve_kernel(const SolveArgs a) {
  if (a.ctrl->stop) return;
  __shared__ SolveKernelSmem s;
  solve_kernel_prologue<6>(a, s, 1.0);
  lio_solve_block(a, s.sm, s.io, s.ctrl);
  __syncthreads();
  if (threadIdx.x == 0) a.ctrl->iter = s.ctrl.iter, a.ctrl->rematch_num = s.ctrl.rematch_num, a.ctrl->stop = s.ctrl.stop;
}

__device__ __forceinline__ void vio_write_stats(const SolveArgs &a, SolveSmem &sm, SolveIO &io) {
  const int tid = threadIdx.x, level = a.level, iteration = a.slot_iter;
  const bool accepted = io.flags[0] != 0, ran = io.flags[2] != 0;
  if (ran && a.vio_stats && level < 8) {
    esikf_vio_stats &S = *a.vio_stats;
    if (accepted && iteration < 8) {
      for (int t = tid; t < 49; t += blockDim.x) S.HTH[level][iteration][t] = sm.A[t];
      for (int t = tid; t < 7; t += blockDim.x) S.HTz[level][iteration][t] = sm.HTz[t];
      for (int t = tid; t < 19; t += blockDim.x) S.solution[level][iteration][t] = sm.sol[t];
    }
    if (tid == 0) {
      if (iteration < 8) S.error_trace[level][iteration] = reinterpret_cast<float *>(io.flags)[4];
      S.iters_per_level[level] = iteration + 1;
      if (accepted) S.accepted_per_level[level] += 1;
      S.total_iters += 1;
    }
  }
}

// One VIO accept/rollback + gain solve (src/vio.cpp:1636-1685) by the calling block; on the last slot also the final
// covariance update (:800). Returns EKF_end of the level. Staged as for lio_solve_block (vec: :1664, gain_setup<7>); a level
// that already ended (EKF_end) comes here on its last slot only, and then only P, the poses and old_state are read.
__device__ __noinline__ bool vio_solve_block(const SolveArgs &a, SolveSmem &sm, SolveIO &io, Ctrl &ctrl) {
  const int tid = threadIdx.x, lane = tid & 31;
  const bool level_done_in = (a.slot_iter == 0) ? false : (ctrl.level_done != 0);   // entering a level: EKF_end = false (vio.cpp:1527)
  const float last_error_in = (a.slot_iter == 0) ? FLT_MAX : ctrl.last_error;       // :1528
  const int has_G_in = ctrl.has_G;
  if (tid < 32) {
    bool accepted = false, ekf_end = level_done_in;
    float error = 0.f, last_error = last_error_in;
    if (!level_done_in) {
      if (a.slot_iter == 0 && lane < 25) io.old[lane] = io.st[lane];  // old_state = *state at level entry (:1523)
      // error = sum(res^2) / n_meas as float (vio.cpp:1636)
      const double sum_sq = io.info[INFO_EXTRA(7)];
      const int n_meas = (int)io.info[INFO_COUNTM(7)];
      error = __fdiv_rn((float)sum_sq, (float)n_meas);
      if (error <= last_error) {  // :1648
        accepted = true;
        if (lane < 25) io.old[lane] = io.st[lane];  // old_state = *state
        last_error = error;
        unpack_info<7>(sm, io, lane);  // H^T H 7x7, H^T z
        double x[7];
        gain_rows<7>(sm, 1.0 / a.img_point_cov, a.solve_mode, lane, x);
        if (a.dbg && tid == 0) a.dbg[0] = globaltimer_ns();
        double g[7];
#pragma unroll
        for (int j = 0; j < 7; j++) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < 7; k++) s += x[k] * sm.A[k * 7 + j];
          g[j] = s;
        }
        if (lane < 19) {
          double s1 = 0.0, s2 = 0.0;
#pragma unroll
          for (int k = 0; k < 7; k++) s1 += x[k] * sm.HTz[k], s2 += g[k] * sm.vec[k];
          sm.sol[lane] = -s1 + sm.vec[lane] - s2;  // :1667
#pragma unroll
          for (int j = 0; j < 7; j++) io.g[lane][j] = g[j];  // G.block<19,7>  (:1665)
        }
        __syncwarp();
        boxplus_warp(io.st, sm.sol, lane);
        if (a.dbg && tid == 0) a.dbg[1] = globaltimer_ns();
        // :1675 (float constants 57.3f / 100.0f / 0.001f promote to double against the double norm)
        ekf_end = (warp_norm3(sm.sol) * (double)57.3f < (double)0.001f) && (warp_norm3(sm.sol + 3) * (double)100.0f < (double)0.001f);
      } else {
        __syncwarp();
        if (lane < 25) io.st[lane] = io.old[lane];  // *state = old_state  (:1679)
        ekf_end = true;
      }
    }
    if (lane == 0) {
      io.flags[0] = accepted, io.flags[1] = ekf_end, io.flags[2] = !level_done_in;
      reinterpret_cast<float *>(io.flags)[3] = last_error;
      reinterpret_cast<float *>(io.flags)[4] = error;
      if (!level_done_in) {
        ctrl.iter += 1;
        ctrl.last_error = last_error;
        if (a.slot_iter == 0) ctrl.accepted_in_level = 0;
        if (accepted) ctrl.has_G = 1, ctrl.accepted_in_level += 1;
      }
      ctrl.level_done = ekf_end;
      if (a.last_slot) ctrl.stop = 1;
    }
  }
  __syncthreads();
  const bool accepted = io.flags[0] != 0, ran = io.flags[2] != 0;
  if (ran && !a.no_publish) {
    for (int t = tid; t < 25; t += blockDim.x) {
      a.state[t] = io.st[t];
      a.old_state[t] = io.old[t];
    }
    if (accepted)
      for (int t = tid; t < 133; t += blockDim.x) a.G[t] = io.g[t / 7][t % 7];
    vio_write_stats(a, sm, io);
  }
  if (a.last_slot && !a.no_publish) {
    // state->cov -= G * state->cov   (vio.cpp:800) with the last accepted G (this slot's if accepted, else the stored one)
    const bool haveG = accepted || has_G_in;
    if (haveG)
      for (int t = tid; t < 361; t += blockDim.x) {
        const int r = t / 19, c = t - 19 * r;
        double s = 0.0;
        for (int j = 0; j < 7; j++) s += (accepted ? io.g[r][j] : __ldcg(a.G + r * 7 + j)) * sm.P[j * 19 + c];
        a.state[S_COV + t] = sm.P[t] - s;
      }
  }
  return io.flags[1] != 0;
}

__global__ void __launch_bounds__(SOLVE_THREADS, 1) vio_solve_kernel(const SolveArgs a) {
  __shared__ SolveKernelSmem s;
  if (solve_kernel_prologue<7>(a, s, 1.0 / a.img_point_cov)) vio_solve_block(a, s.sm, s.io, s.ctrl);
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned bc = a.ctrl->block_counter;
    *a.ctrl = s.ctrl;
    a.ctrl->block_counter = bc;
  }
}

}  // namespace esikf
