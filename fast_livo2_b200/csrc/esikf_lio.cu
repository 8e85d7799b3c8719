// LIO kernels of the B200 ESIKF update (sm_100a).
//
//   lio_precompute_kernel : per-frame calcBodyCov + cross-matrix vector     (reference src/voxel_map.cpp:15-34, 349-360)
//   plane_compact_kernel  : 256-byte map plane -> 144-byte record the residual build consumes (map upload / patch time)
//   lio_residual_kernel   : one ESIKF iteration's residual / Jacobian build (src/voxel_map.cpp:376-390 TransformLidar + point
//                           covariance, :643-786 voxel probe + plane association, :414-458 Jacobian / R^-1) fused with the
//                           H^T R^-1 H, H^T R^-1 z reduction (:464-466). No PointToPlane is ever materialised.
//
// Mapping: one thread per LiDAR point, 22 warps per CTA, one CTA per SM (148 x 704 = 104 k points resident in one round).
// Every lane owns a 304-byte shared-memory slot for the whole update: the plane record of its point's voxel (brought in by
// ONE cp.async.bulk per lane, completion counted on a per-warp mbarrier), the point's body covariance, and everything
// about the (point, plane) pair that does not change from one iteration to the next:
//   * the voxel key / candidate range (no hash probe while the point stays in its voxel),
//   * u^T P_rot u + n^T P_pos n, the state-covariance part of n^T var n (state_.cov is constant inside the loop, :377-389),
//   * R_inv, which the reference evaluates with the PRIOR pose (:425-449) and therefore repeats unchanged every iteration.
// What is left per iteration is p_w, the two gates, a 3x3 quadratic form and the Jacobian row: ~110 fp64 operations out of
// shared memory instead of ~450 plus three dependent global round trips. The warp is the cooperation unit for the rest:
// the rare extra candidates of sub-divided root voxels of ALL lanes are evaluated lane-parallel in one pass, and the
// per-warp contraction sum_i a_i (w_i a_i)^T, a = [H_i(6), z_i, 1], runs on the fp64 tensor-core path
// (mma.sync.m8n8k4.f64, SASS DMMA). Partial sums are combined in a fixed order (warp -> CTA -> grid): bit-reproducible.
#include "esikf_dev.cuh"

namespace esikf {

// Cold paths (extras of sub-divided voxels, neighbour voxel, record staging, R_inv) inline or out of line: measured on config 2,
// inlining is faster (LIO update 129.5 us against 145.4 us: the call sequences and the callees' own spills cost more than the
// register pressure they take off the hot path); -DLIO_COLD=__noinline__ rebuilds the other variant.
#ifndef LIO_COLD
#define LIO_COLD __forceinline__
#endif
#ifndef LIO_FULL_REC
#define LIO_FULL_REC 0  // cold candidates: head first, covariance part after the range gate (0, default) or the whole record in one round trip (1). Measured on config 2: 123.3 us against 132.0 us per LIO update — the 18 extra live registers of the one-trip form cost more in spills than the saved L2 round trip (profiles/loop_modes_r02_ab_cold_paths.txt)
#endif
#define LIO_THREADS 704  // 22 warps, one CTA per SM: 148 x 704 = 104k points in a single round
#define LIO_WARPS (LIO_THREADS / 32)

struct LioKernelArgs {
  const float *pts;          // [n_total][3] body-frame scan
  const double *pre;         // SoA [9][pre_stride]: cross vector c(3) | body cov xx xy xz yy yz zz
  int pre_stride;
  int partial_stride;
  int begin, count;          // this rank's shard
  const double *state;       // current iterate (device, packed)
  const double *prop;        // state_propagat
  const HashSlot *slots;
  uint32_t hash_mask;
  const PlaneRec *recs;      // compact plane records, DFS order per root voxel
  double extR[9], extT[3];
  double voxel_size;         // double voxel size used for the key (voxel_map.cpp:646,668)
  double inv_voxel_size;     // 1 / voxel_size, used when exact
  int inv_voxel_exact;
  float voxel_size_f;        // float voxel size that positioned the roots (voxel_map.cpp:534,578-581)
  double sigma_num;
  int32_t *match_plane;      // [n_total]
  int32_t *normal_plane;     // [n_total] sticky
  float *dis_to_plane;       // [n_total]
  double *partials;          // [NE][partial_stride]
  double *info;              // [NE_MAX]
  Ctrl *ctrl;
  int init_normal;           // first iteration of an update: unmatched points get normal_plane = -1 (pv.normal = 0)
  int stage_mode;            // 0: cp.async.bulk per lane (default), 1: coalesced half-warp __ldg copies (measurement variant)
};

// What the out-of-line cold paths need of the kernel arguments, passed BY VALUE: taking the address of the kernel-parameter
// struct would move it (and every hot-path read of it) from the constant bank to local memory.
struct LioCold {
  const PlaneRec *recs;
  const HashSlot *slots;
  uint32_t hash_mask;
  float voxel_size_f;
  double sigma_num;
  double voxel_size, inv_voxel_size;
  int inv_voxel_exact, stage_mode;
  double extR[9], extT[3];
};

__device__ __forceinline__ double dot3_rn(double a0, double a1, double a2, double b0, double b1, double b2) {
  return __dadd_rn(__dadd_rn(__dmul_rn(a0, b0), __dmul_rn(a1, b1)), __dmul_rn(a2, b2));
}
// index of (i,j) in the row-major upper triangle of a 6x6
__host__ __device__ constexpr int tri6(int i, int j) { return (i <= j) ? (i * 6 - (i * (i - 1)) / 2 + (j - i)) : (j * 6 - (j * (j - 1)) / 2 + (i - j)); }

__device__ __forceinline__ double quad3_sym(const double *v, double n0, double n1, double n2) {
  // n^T V n with V symmetric (xx xy xz yy yz zz), evaluated as (n^T V) n
  const double t0 = n0 * v[0] + n1 * v[1] + n2 * v[2];
  const double t1 = n0 * v[1] + n1 * v[3] + n2 * v[4];
  const double t2 = n0 * v[2] + n1 * v[4] + n2 * v[5];
  return t0 * n0 + t1 * n1 + t2 * n2;
}
__device__ __forceinline__ double quad3_full(const double *P, double u0, double u1, double u2) {
  // u^T P u with P a row-major 3x3
  return (u0 * P[0] + u1 * P[3] + u2 * P[6]) * u0 + (u0 * P[1] + u1 * P[4] + u2 * P[7]) * u1 + (u0 * P[2] + u1 * P[5] + u2 * P[8]) * u2;
}

// ---------------------------------------------------------------------------------------------------------------------
// Per-frame precompute: calcBodyCov (voxel_map.cpp:15-34) and the cross-matrix vector extR*p+extT (:356-359).
__global__ void lio_precompute_kernel(const float *__restrict__ pts, int n, double *__restrict__ pre, int pre_stride,
                                      const double *__restrict__ ext, float dept_err, float beam_err) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double px = pts[3 * i], py = pts[3 * i + 1], pz = pts[3 * i + 2];
  if (pz == 0) pz = 0.001;  // :352  (calcBodyCov's own 0 -> 1e-4 fix at :17 can then never trigger)
  float range = (float)sqrt(px * px + py * py + pz * pz);
  float range_var = dept_err * dept_err;
  double sdv = sin((double)beam_err * 0.017453293);  // PCL DEG2RAD
  double dv = sdv * sdv;
  double nrm = sqrt(px * px + py * py + pz * pz);
  double dx = px / nrm, dy = py / nrm, dz = pz / nrm;
  double b1x = 1.0, b1y = 1.0, b1z = -(dx + dy) / dz;
  double n1 = sqrt(b1x * b1x + b1y * b1y + b1z * b1z);
  b1x /= n1, b1y /= n1, b1z /= n1;
  double b2x = b1y * dz - b1z * dy, b2y = b1z * dx - b1x * dz, b2z = b1x * dy - b1y * dx;  // base_vector1.cross(direction)
  double n2 = sqrt(b2x * b2x + b2y * b2y + b2z * b2z);
  b2x /= n2, b2y /= n2, b2z /= n2;
  // A = range * [d]x * [b1 b2]   (3x2)
  double r = (double)range;
  double a00 = r * (-dz * b1y + dy * b1z), a01 = r * (-dz * b2y + dy * b2z);
  double a10 = r * (dz * b1x - dx * b1z), a11 = r * (dz * b2x - dx * b2z);
  double a20 = r * (-dy * b1x + dx * b1y), a21 = r * (-dy * b2x + dx * b2y);
  double rv = (double)range_var;
  double *o = pre + i;
  const size_t ns = (size_t)pre_stride;
  // cross vector
  o[0 * ns] = ext[0] * px + ext[1] * py + ext[2] * pz + ext[9];
  o[1 * ns] = ext[3] * px + ext[4] * py + ext[5] * pz + ext[10];
  o[2 * ns] = ext[6] * px + ext[7] * py + ext[8] * pz + ext[11];
  // cov = d rv d^T + A dv A^T  (symmetric; upper triangle stored)
  o[3 * ns] = dx * rv * dx + dv * (a00 * a00 + a01 * a01);
  o[4 * ns] = dx * rv * dy + dv * (a00 * a10 + a01 * a11);
  o[5 * ns] = dx * rv * dz + dv * (a00 * a20 + a01 * a21);
  o[6 * ns] = dy * rv * dy + dv * (a10 * a10 + a11 * a11);
  o[7 * ns] = dy * rv * dz + dv * (a10 * a20 + a11 * a21);
  o[8 * ns] = dz * rv * dz + dv * (a20 * a20 + a21 * a21);
}

// 256-byte plane (VoxelPlane as uploaded) -> compact record. ids == nullptr: planes [0, n); else the listed plane ids.
// plane_var_ is consumed through its upper triangle, (i, j) and (j, i) read the same value.
__global__ void plane_compact_kernel(const esikf_plane *__restrict__ planes, const int32_t *__restrict__ ids, int n, PlaneRec *__restrict__ recs) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int id = ids ? ids[k] : k;
  PlaneRec r;
  compact_plane(planes[id], r);
  recs[id] = r;
}

// ---------------------------------------------------------------------------------------------------------------------
struct Cand {
  double prob;
  int idx;
  float dis;  // signed n.p + d narrowed to float (PointToPlane::dis_to_plane_, voxel_map.cpp:753)
};

// Lane slot layout (doubles). [0, 18) is the PlaneRec image (bulk-copied); the row part feeds the tensor-core contraction.
// 304 B = 19 x 16 B: 16-byte aligned for the bulk copy and conflict-free for 128-bit accesses at lane stride — every
// hot-path access below is a double2.
#define SLOT_D 38
enum { SL_C = 0, SL_N = 3, SL_PAA = 6, SL_B = 12, SL_CNN = 15, SL_DR = 16, SL_OUT = 17, SL_BC = 18, SL_SPP = 24, SL_WGT = 25, SL_KEY = 26, SL_META = 27, SL_ROW = 28, SL_PT = 37 };
// SL_OUT : {i32 match_plane, i32 normal_plane} of the last iteration (the bulk copy writes PlaneRec::pad here: set after staging)
// SL_META: {u32 candidate count of the cached voxel (LIO_ABSENT: no such voxel), i32 plane the cached R_inv belongs to}
// SL_ROW : A0 A1 A2 n0 n1 n2 z w {f32 signed dis_to_plane, f32 raw point z}
// SL_PT  : {f32 raw point x, f32 raw point y}
// Everything a lane carries from one iteration to the next lives here, not in registers: the hot path has 80 of them.
#define LIO_ABSENT 0xFFFFFFFFu
__device__ __forceinline__ void slot_point(const double *slot, float &px, float &py, float &pz) {
  const float2 xy = *reinterpret_cast<const float2 *>(slot + SL_PT);
  px = xy.x, py = xy.y, pz = reinterpret_cast<const float *>(slot + SL_ROW + 8)[1];
}

// shared-memory layout of the residual kernel
struct __align__(128) LioSmem {
  double rec[LIO_WARPS][32][SLOT_D];
  double R[9], t[3], Ptt[9], Ppp[9];      // current state
  double Rp[9], tp[3], Mp[9];             // prior pose, Mp = Rp * extR
  LioCold cold;                           // what the out-of-line cold paths read of the kernel arguments
  unsigned long long mbar[LIO_WARPS];     // one bulk-copy barrier per warp
  ReduceSmem<LIO_WARPS> red;
  unsigned char fs_raw[8704];             // the CTA's resident solve state (FusedSolveSmem) in the persistent kernel
};

// What a lane keeps about ITS point across the iterations of a persistent update (registers); the rest is in its slot.
struct LaneCache {
  int staged_idx;    // plane whose record is resident in the slot (-1: none)
  bool have_pt;      // pi / body covariance loaded
  bool key_valid;    // slot holds the voxel key + candidate count of the last probe
  bool out_valid;    // the slot holds this lane's per-point outputs
  unsigned mphase;   // parity of the warp's bulk-copy barrier
};
__device__ __forceinline__ void lane_cache_reset(LaneCache &lc) {
  lc.staged_idx = -1, lc.have_pt = false, lc.key_valid = false;
}
__device__ __forceinline__ void lane_cache_init(LaneCache &lc) {
  lane_cache_reset(lc);
  lc.mphase = 0;
  lc.out_valid = false;
}

// The pose constants of the residual build, into shared memory by threads 0..11; the caller's CTA barrier publishes them.
// The state comes from global memory in the per-iteration kernel and from the CTA's resident copy in the persistent one.
// Prior pose (voxel_map.cpp:425-428) and Mp = Rp * extR (state_propagat.rot_end * extR_, :445).
__device__ __forceinline__ void lio_prior_consts(LioSmem &sm, const LioKernelArgs &a) {
  const int tid = threadIdx.x;
  if (tid < 9) {
    const int r = tid / 3, c = tid % 3;
    sm.Rp[tid] = a.prop[S_R + tid];
    double s = 0;
    for (int k = 0; k < 3; k++) s += a.prop[S_R + r * 3 + k] * a.extR[k * 3 + c];
    sm.Mp[tid] = s;
  } else if (tid < 12) {
    sm.tp[tid - 9] = a.prop[S_P + tid - 9];
  }
}
// Covariance blocks of pv.var (:377-378) out of the 19 x 19 covariance P.
__device__ __forceinline__ void lio_cov_consts(LioSmem &sm, const double *P) {
  const int tid = threadIdx.x;
  if (tid < 9) {
    const int r = tid / 3, c = tid % 3;
    sm.Ptt[tid] = P[r * 19 + c];
    sm.Ppp[tid] = P[(3 + r) * 19 + (3 + c)];
  }
}
// Current pose R, t out of the packed state.
__device__ __forceinline__ void lio_pose_consts(LioSmem &sm, const double *st) {
  const int tid = threadIdx.x;
  if (tid < 9) {
    sm.R[tid] = st[S_R + tid];
  } else if (tid < 12) {
    sm.t[tid - 9] = st[S_P + tid - 9];
  }
}

__device__ __forceinline__ bool probe(const HashSlot *__restrict__ slots, uint32_t mask, long long kx, long long ky, long long kz,
                                      uint32_t &first, uint32_t &count) {
  if (!key_in_range(kx, ky, kz)) return false;
  unsigned long long key = pack_key(kx, ky, kz);
  uint32_t s = hash_key(key) & mask;
  for (;;) {
    ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(slots + s));
    if (v.x == key) {
      first = (uint32_t)(v.y & 0xffffffffull);
      count = (uint32_t)(v.y >> 32);
      return true;
    }
    if (v.x == ESIKF_KEY_EMPTY) return false;
    s = (s + 1) & mask;
  }
}

// Head of a plane record (shared-memory slot or global record, 16-byte aligned): centre, normal, d, radius.
struct RecHead {
  double c0, c1, c2, n0, n1, n2;
  float d, radius;
};
__device__ __forceinline__ RecHead load_head(const double *__restrict__ q) {
  const double2 *__restrict__ q2 = reinterpret_cast<const double2 *>(q);
  const double2 a0 = q2[0], a1 = q2[1], a2 = q2[2];
  const float2 dr = *reinterpret_cast<const float2 *>(q + SL_DR);
  RecHead h;
  h.c0 = a0.x, h.c1 = a0.y, h.c2 = a1.x, h.n0 = a1.y, h.n1 = a2.x, h.n2 = a2.y, h.d = dr.x, h.radius = dr.y;
  return h;
}

// The float-rounded quantities that gate the association (voxel_map.cpp:723-731), evaluated without FMA contraction, left
// to right, like the reference: signed distance, |distance| and the in-plane range test.
struct Gate1 {
  double sd;
  float dis_to_plane;
  double e0, e1, e2;  // c - p_w
  bool pass;
};
__device__ __forceinline__ Gate1 gate_range(const RecHead &h, const double pw[3]) {
  Gate1 g;
  g.sd = __dadd_rn(dot3_rn(h.n0, h.n1, h.n2, pw[0], pw[1], pw[2]), (double)h.d);
  g.dis_to_plane = (float)fabs(g.sd);
  g.e0 = h.c0 - pw[0], g.e1 = h.c1 - pw[1], g.e2 = h.c2 - pw[2];
  const float dis_to_center = (float)dot3_rn(g.e0, g.e1, g.e2, g.e0, g.e1, g.e2);
  const float range_dis = sqrtf(__fsub_rn(dis_to_center, __fmul_rn(g.dis_to_plane, g.dis_to_plane)));
  g.pass = (double)range_dis <= 3.0 * (double)h.radius;  // NaN fails, as in the reference
  return g;
}
// J plane_var J^T for J = [p - c, -n] (:733-735) from the compact record: e^T Paa e + 2 e^T b + cnn, e = c - p.
__device__ __forceinline__ double sigma_plane(const double *__restrict__ q, double e0, double e1, double e2) {
  const double2 *__restrict__ q2 = reinterpret_cast<const double2 *>(q);
  const double2 p0 = q2[3], p1 = q2[4], p2 = q2[5], b01 = q2[6], b2c = q2[7];  // paa xx xy | xz yy | yz zz ; b0 b1 ; b2 cnn
  const double t0 = e0 * p0.x + e1 * p0.y + e2 * p1.x;
  const double t1 = e0 * p0.y + e1 * p1.y + e2 * p2.x;
  const double t2 = e0 * p1.x + e1 * p2.x + e2 * p2.y;
  return (t0 * e0 + t1 * e1 + t2 * e2) + 2.0 * (e0 * b01.x + e1 * b01.y + e2 * b2c.x) + b2c.y;
}
// m^T body_cov m, body covariance (xx xy xz yy yz zz) at bc (16-byte aligned, a slot's SL_BC)
__device__ __forceinline__ double quad_bc(const double *bc, double m0, double m1, double m2) {
  const double2 *b2 = reinterpret_cast<const double2 *>(bc);
  const double2 v0 = b2[0], v1 = b2[1], v2 = b2[2];  // xx xy | xz yy | yz zz
  const double t0 = m0 * v0.x + m1 * v0.y + m2 * v1.x;
  const double t1 = m0 * v0.y + m1 * v1.y + m2 * v2.x;
  const double t2 = m0 * v1.x + m1 * v2.x + m2 * v2.y;
  return t0 * m0 + t1 * m1 + t2 * m2;
}
// State-covariance part of n^T pv.var n (:385-388): pv.var = R body_cov R^T + [c]x P_rot [c]x^T + P_pos, so
//   n^T var n = m^T body_cov m + u^T P_rot u + n^T P_pos n,   m = R^T n,  u = c x n  (c = the cross-matrix vector).
__device__ __forceinline__ double spp_of(const RecHead &h, double cx, double cy, double cz, const double *Ptt, const double *Ppp) {
  const double u0 = cy * h.n2 - cz * h.n1, u1 = cz * h.n0 - cx * h.n2, u2 = cx * h.n1 - cy * h.n0;
  return quad3_full(Ptt, u0, u1, u2) + quad3_full(Ppp, h.n0, h.n1, h.n2);
}
__device__ __forceinline__ void rot_t_n(const double *R, const RecHead &h, double &m0, double &m1, double &m2) {
  m0 = R[0] * h.n0 + R[3] * h.n1 + R[6] * h.n2, m1 = R[1] * h.n0 + R[4] * h.n1 + R[7] * h.n2, m2 = R[2] * h.n0 + R[5] * h.n1 + R[8] * h.n2;
}
// this_prob of :740 — only needed to arbitrate between several candidates that pass both gates
__device__ __forceinline__ double prob_of(double sigma_l, float dis_to_plane) {
  return 1.0 / sqrt(sigma_l) * exp(-0.5 * (double)dis_to_plane * (double)dis_to_plane / sigma_l);
}

// build_single_residual's plane branch (:721-768) for a candidate that is NOT the lane's resident record (extra candidates
// of sub-divided voxels, neighbour voxels): everything from scratch. bc: body covariance (6), c*: cross-matrix vector.
struct EvalOut {
  bool pass;
  double sigma_l;
  float dis, dis_to_plane;
};
__device__ __forceinline__ EvalOut eval_cold(const double *__restrict__ q, const double pw[3], const double *bc, double cx, double cy, double cz,
                                             const LioSmem &sm, double sigma_num) {
  EvalOut o;
  o.pass = false, o.sigma_l = 0.0, o.dis = 0.f, o.dis_to_plane = 0.f;
#if !LIO_FULL_REC
  {
    const RecHead h = load_head(q);
    const Gate1 g = gate_range(h, pw);
    if (g.pass) {
      double m0, m1, m2;
      rot_t_n(sm.R, h, m0, m1, m2);
      const double sigma_l = sigma_plane(q, g.e0, g.e1, g.e2) + quad_bc(bc, m0, m1, m2) + spp_of(h, cx, cy, cz, sm.Ptt, sm.Ppp);
      if ((double)g.dis_to_plane < sigma_num * sqrt(sigma_l)) o.pass = true, o.sigma_l = sigma_l, o.dis = (float)g.sd, o.dis_to_plane = g.dis_to_plane;
    }
    return o;
  }
#endif
  // the whole 144-byte record in ONE round trip (these records come from global memory: a second, dependent trip for the
  // covariance part after the range gate would double the latency of the pass)
  const double2 *__restrict__ q2 = reinterpret_cast<const double2 *>(q);
  const double2 r0 = __ldg(q2), r1 = __ldg(q2 + 1), r2 = __ldg(q2 + 2), r3 = __ldg(q2 + 3), r4 = __ldg(q2 + 4), r5 = __ldg(q2 + 5), r6 = __ldg(q2 + 6), r7 = __ldg(q2 + 7),
                r8 = __ldg(q2 + 8);
  RecHead h;
  h.c0 = r0.x, h.c1 = r0.y, h.c2 = r1.x, h.n0 = r1.y, h.n1 = r2.x, h.n2 = r2.y;
  h.d = __int_as_float((int)(__double_as_longlong(r8.x) & 0xffffffffll)), h.radius = __int_as_float((int)(__double_as_longlong(r8.x) >> 32));
  const Gate1 g = gate_range(h, pw);
  if (g.pass) {
    double m0, m1, m2;
    rot_t_n(sm.R, h, m0, m1, m2);
    // sigma_plane on the registers: paa = r3 r4 r5 (xx xy | xz yy | yz zz), b = r6.x r6.y r7.x, cnn = r7.y
    const double t0 = g.e0 * r3.x + g.e1 * r3.y + g.e2 * r4.x;
    const double t1 = g.e0 * r3.y + g.e1 * r4.y + g.e2 * r5.x;
    const double t2 = g.e0 * r4.x + g.e1 * r5.x + g.e2 * r5.y;
    const double sp = (t0 * g.e0 + t1 * g.e1 + t2 * g.e2) + 2.0 * (g.e0 * r6.x + g.e1 * r6.y + g.e2 * r7.x) + r7.y;
    const double sigma_l = sp + quad_bc(bc, m0, m1, m2) + spp_of(h, cx, cy, cz, sm.Ptt, sm.Ppp);
    if ((double)g.dis_to_plane < sigma_num * sqrt(sigma_l)) o.pass = true, o.sigma_l = sigma_l, o.dis = (float)g.sd, o.dis_to_plane = g.dis_to_plane;
  }
  return o;
}

// Layout of the (owner lane, extra candidate) pairs of a warp: the pairs of all pending lanes are laid out consecutively and
// dealt one per lane per chunk, so the scattered plane-record reads of every pending point overlap instead of being paid
// once per pending lane (the slowest warp of the slowest CTA sets the grid barrier).
struct PairLayout {
  unsigned mask;  // pending lanes
  int npairs, excl, total;
};
__device__ __forceinline__ PairLayout pair_layout(bool pending, uint32_t count, int lane) {
  PairLayout L;
  L.mask = __ballot_sync(0xffffffffu, pending);
  L.npairs = pending ? (int)count - 1 : 0;
  int scan = L.npairs;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, scan, d);
    if (lane >= d) scan += t;
  }
  L.total = __shfl_sync(0xffffffffu, scan, 31);
  L.excl = scan - L.npairs;
  return L;
}
__device__ __forceinline__ void pair_of(const PairLayout &L, int k, int &owner, int &cand) {
  owner = 0, cand = 0;
  for (unsigned m = L.mask; m; m &= m - 1) {
    const int jl = __ffs(m) - 1;
    const int ej = __shfl_sync(0xffffffffu, L.excl, jl), nj = __shfl_sync(0xffffffffu, L.npairs, jl);
    if (k >= ej && k < ej + nj) owner = jl, cand = k - ej + 1;
  }
}

// Pass 1 over the extra candidates (sub-divided root voxels) of ALL pending lanes of the warp: which of them pass both
// gates. Per pending lane: npass = number of passing extras, (fidx, fdis) = the first of them in DFS order. No
// probabilities: a point whose candidates pass at most once in total needs none (any passing candidate has this_prob > 0
// and wins, :741-768); only points with two or more passing candidates go through warp_eval_extras_prob.
__device__ __forceinline__ void warp_eval_extras_count(const LioCold &a, const LioSmem &sm, const double (*wslots)[SLOT_D], bool pending, const double pw[3],
                                                       double cx, double cy, double cz, uint32_t first, uint32_t count, int lane, int &npass, int &fidx, float &fdis) {
  npass = 0, fidx = -1, fdis = 0.f;
  const PairLayout L = pair_layout(pending, count, lane);
  if (!L.mask) return;
  for (int base = 0; base < L.total; base += 32) {
    const int k = base + lane;
    int owner, cand;
    pair_of(L, k, owner, cand);
    const bool have = k < L.total;
    double opw[3];
#pragma unroll
    for (int c = 0; c < 3; c++) opw[c] = __shfl_sync(0xffffffffu, pw[c], owner);
    const double ocx = __shfl_sync(0xffffffffu, cx, owner), ocy = __shfl_sync(0xffffffffu, cy, owner), ocz = __shfl_sync(0xffffffffu, cz, owner);
    const uint32_t ofirst = __shfl_sync(0xffffffffu, first, owner);
    bool pass = false;
    float dis = 0.f;
    if (have) {
      const EvalOut e = eval_cold(reinterpret_cast<const double *>(a.recs + ofirst + cand), opw, &wslots[owner][SL_BC], ocx, ocy, ocz, sm, a.sigma_num);
      pass = e.pass, dis = e.dis;
    }
    const int myidx = (int)(ofirst + cand);
    for (unsigned m = L.mask; m; m &= m - 1) {
      const int jl = __ffs(m) - 1;
      const unsigned pm = __ballot_sync(0xffffffffu, have && owner == jl && pass);
      const int src = pm ? __ffs(pm) - 1 : 0;  // lowest lane = lowest candidate index of this chunk
      const int sidx = __shfl_sync(0xffffffffu, myidx, src);
      const float sdis = __shfl_sync(0xffffffffu, dis, src);
      if (lane == jl && pm) {
        if (fidx < 0) fidx = sidx, fdis = sdis;
        npass += __popc(pm);
      }
    }
  }
}

// Pass 2, only for lanes with two or more passing candidates: winner = arg-max probability with lowest-index tie break,
// merged with `best` (the first candidate's result) by strict '>' — exactly the order-dependent rule of the recursion
// (voxel_map.cpp:741: the first of equal probabilities is kept).
__device__ __forceinline__ void warp_eval_extras_prob(const LioCold &a, const LioSmem &sm, const double (*wslots)[SLOT_D], bool pending, const double pw[3],
                                                      double cx, double cy, double cz, uint32_t first, uint32_t count, int lane, Cand &best) {
  const PairLayout L = pair_layout(pending, count, lane);
  if (!L.mask) return;
  Cand acc;
  acc.prob = -1.0, acc.idx = -1, acc.dis = 0.f;
  for (int base = 0; base < L.total; base += 32) {
    const int k = base + lane;
    int owner, cand;
    pair_of(L, k, owner, cand);
    const bool have = k < L.total;
    double opw[3];
#pragma unroll
    for (int c = 0; c < 3; c++) opw[c] = __shfl_sync(0xffffffffu, pw[c], owner);
    const double ocx = __shfl_sync(0xffffffffu, cx, owner), ocy = __shfl_sync(0xffffffffu, cy, owner), ocz = __shfl_sync(0xffffffffu, cz, owner);
    const uint32_t ofirst = __shfl_sync(0xffffffffu, first, owner);
    Cand my;
    my.prob = -1.0, my.idx = 0x7fffffff, my.dis = 0.f;
    if (have) {
      const EvalOut e = eval_cold(reinterpret_cast<const double *>(a.recs + ofirst + cand), opw, &wslots[owner][SL_BC], ocx, ocy, ocz, sm, a.sigma_num);
      if (e.pass) my.prob = prob_of(e.sigma_l, e.dis_to_plane), my.idx = (int)(ofirst + cand), my.dis = e.dis;
    }
    for (unsigned m = L.mask; m; m &= m - 1) {
      const int jl = __ffs(m) - 1;
      const bool mine = have && owner == jl && my.idx != 0x7fffffff;
      double rp = mine ? my.prob : -1.0;
      int ri = mine ? my.idx : 0x7fffffff;
      float rd = mine ? my.dis : 0.f;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const double op = __shfl_xor_sync(0xffffffffu, rp, off);
        const int oi = __shfl_xor_sync(0xffffffffu, ri, off);
        const float od = __shfl_xor_sync(0xffffffffu, rd, off);
        if (op > rp || (op == rp && oi < ri)) rp = op, ri = oi, rd = od;
      }
      // chunks are visited in increasing candidate order: a later chunk only replaces on strictly larger probability
      if (lane == jl && ri != 0x7fffffff && rp > acc.prob) acc.prob = rp, acc.idx = ri, acc.dis = rd;
    }
  }
  if (pending && acc.idx >= 0 && acc.prob > best.prob) best = acc;
}

// All candidates of one root voxel for the lanes that have one (`act`): the first candidate's result is (pass0, sigma0,
// sd0, dtp0) — evaluated by the caller, from the slot or cold —, the extras are counted lane-parallel; probabilities are
// evaluated only where two or more candidates pass. On return best_idx / best_dis hold the winner (or -1).
__device__ LIO_COLD void resolve_voxel(const LioCold &a, const LioSmem &sm, const double (*wslots)[SLOT_D], bool act, const double pw[3], double cx, double cy,
                                              double cz, uint32_t first, uint32_t count, bool pass0, double sigma0, float dis0, float dtp0, int lane, int &best_idx,
                                              float &best_dis) {
  const bool pend = act && count > 1;
  int npass, fidx;
  float fdis;
  warp_eval_extras_count(a, sm, wslots, pend, pw, cx, cy, cz, first, count, lane, npass, fidx, fdis);
  const int total = (act && pass0 ? 1 : 0) + npass;
  if (act) {
    if (pass0) best_idx = (int)first, best_dis = dis0;
    else if (total >= 1) best_idx = fidx, best_dis = fdis;
  }
  const bool slow = pend && total >= 2;
  if (__any_sync(0xffffffffu, slow)) {
    Cand best;
    best.prob = 0.0, best.idx = -1, best.dis = 0.f;
    if (slow && pass0) best.prob = prob_of(sigma0, dtp0), best.idx = (int)first, best.dis = dis0;
    warp_eval_extras_prob(a, sm, wslots, slow, pw, cx, cy, cz, first, count, lane, best);
    if (slow) best_idx = best.idx, best_dis = best.dis;
  }
}

// p_imu = extR p + extT (TransformLidar, voxel_map.cpp:524). No FMA contraction: the chain ends in the float rounding of p_w,
// which decides the voxel key.
__device__ __forceinline__ void p_imu(const double *extR, const double *extT, float fx, float fy, float fz, double &pi0, double &pi1, double &pi2) {
  const double px = fx, py = fy, pz = fz;
  pi0 = __dadd_rn(dot3_rn(extR[0], extR[1], extR[2], px, py, pz), extT[0]);
  pi1 = __dadd_rn(dot3_rn(extR[3], extR[4], extR[5], px, py, pz), extT[1]);
  pi2 = __dadd_rn(dot3_rn(extR[6], extR[7], extR[8], px, py, pz), extT[2]);
}
// cross-matrix vector of the point (voxel_map.cpp:352-359): extR p + extT with z = 0.001 when the raw z is 0
__device__ __forceinline__ void cross_vec(const double *extR, const double *extT, float fx, float fy, float fz, double &cx, double &cy, double &cz) {
  p_imu(extR, extT, fx, fy, fz, cx, cy, cz);
  if (fz == 0.f) cx += extR[2] * 0.001, cy += extR[5] * 0.001, cz += extR[8] * 0.001;
}
// voxel coordinate of one axis (voxel_map.cpp:665-671): float quotient, "-1 if negative". When 1/voxel_size is exact (a power
// of two: 0.5, 2.0, ...) the multiply gives the bit-identical quotient without the slow fp64 division.
__device__ __forceinline__ float voxel_coord(double pw, double voxel_size, double inv_voxel_size, int exact) {
  float loc = exact ? (float)__dmul_rn(pw, inv_voxel_size) : (float)__ddiv_rn(pw, voxel_size);
  if (loc < 0) loc = (float)__dadd_rn((double)loc, -1.0);
  return loc;
}

// The cold paths are out of line and take few, narrow arguments (p_w is a float triple by construction, everything else
// comes from shared memory): their register needs must not weigh on the hot path, which has 80 registers per thread.
struct AssocOut {
  int idx;
  float dis;
};
// Cold part of the association: the extras of sub-divided home voxels, then one neighbour voxel for the lanes whose home
// voxel gave nothing (voxel_map.cpp:680-691). loc is in voxel units, centre / quarter length in metres: reproduced
// literally. Called by the whole warp. flags: 1 = extras pending, 2 = home voxel exists, 4 = its first candidate passed.
__device__ LIO_COLD AssocOut lio_cold_assoc(const LioSmem &sm, int warp, int lane, unsigned flags, float pwx, float pwy, float pwz, uint32_t first, uint32_t count,
                                            double sigma0, float dis0, float dtp0) {
  const LioCold &a = sm.cold;
  const double *slot = &sm.rec[warp][lane][0];
  float px, py, pz;
  slot_point(slot, px, py, pz);
  const bool pend1 = flags & 1u, found_home = flags & 2u, pass0 = flags & 4u;
  const double pw[3] = {(double)pwx, (double)pwy, (double)pwz};
  double cx, cy, cz;
  cross_vec(a.extR, a.extT, px, py, pz, cx, cy, cz);
  int bi = (pass0 && count == 1) ? (int)first : -1;
  float bd = (pass0 && count == 1) ? dis0 : 0.f;
  resolve_voxel(a, sm, sm.rec[warp], pend1, pw, cx, cy, cz, first, count, pass0, sigma0, dis0, dtp0, lane, bi, bd);
  uint32_t f2 = 0, c2 = 0;
  bool found2 = false;
  EvalOut e2;
  e2.pass = false, e2.sigma_l = 0.0, e2.dis = 0.f, e2.dis_to_plane = 0.f;
  if (found_home && bi < 0) {
    const double vsf = (double)a.voxel_size_f;
    const double ql = (double)(a.voxel_size_f / 4.0f);
    long long key[3], nk[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const float loc = voxel_coord(pw[j], a.voxel_size, a.inv_voxel_size, a.inv_voxel_exact);
      key[j] = nk[j] = (long long)loc;
      const double center = (0.5 + (double)key[j]) * vsf;
      if ((double)loc > center + ql) nk[j] = key[j] + 1;
      else if ((double)loc < center - ql) nk[j] = key[j] - 1;
    }
    found2 = probe(a.slots, a.hash_mask, nk[0], nk[1], nk[2], f2, c2) && c2 > 0;
    if (found2) e2 = eval_cold(reinterpret_cast<const double *>(a.recs + f2), pw, slot + SL_BC, cx, cy, cz, sm, a.sigma_num);
  }
  if (__any_sync(0xffffffffu, found2)) resolve_voxel(a, sm, sm.rec[warp], found2, pw, cx, cy, cz, f2, c2, e2.pass, e2.sigma_l, e2.dis, e2.dis_to_plane, lane, bi, bd);
  AssocOut o;
  o.idx = bi, o.dis = bd;
  return o;
}

// Cold: bring the first candidate record of the lanes' (new) voxels into their slots and evaluate the record-dependent
// invariant u^T P_rot u + n^T P_pos n. Called by the whole warp when at least one lane wants a record.
__device__ LIO_COLD void lio_cold_stage(LioSmem &sm, int warp, int lane, bool want, int cand0, unsigned wmask, unsigned mphase) {
  const LioCold &a = sm.cold;
  double *slot = &sm.rec[warp][lane][0];
  const double keep_out = slot[SL_OUT];  // the record image covers this word
  if (a.stage_mode == 0) {
    // one bulk copy (TMA engine) per lane on the warp's mbarrier; the slot may have been read through the generic proxy before
    unsigned long long *bar = &sm.mbar[warp];
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) mbar_arrive_expect_tx(bar, (unsigned)sizeof(PlaneRec) * __popc(wmask));
    __syncwarp();
    if (want) bulk_g2s(slot, a.recs + cand0, (unsigned)sizeof(PlaneRec), bar);
    mbar_wait(bar, mphase & 1u);
  } else {
    // measurement variant: coalesced half-warp copies, 16 B per lane, two records per instruction
    const int half = lane >> 4, sub = lane & 15;
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
      const int src = j + half;
      const int pidx = __shfl_sync(0xffffffffu, want ? cand0 : -1, src);
      if (pidx >= 0 && sub < 9) {
        const double2 v = __ldg(reinterpret_cast<const double2 *>(a.recs + pidx) + sub);
        *reinterpret_cast<double2 *>(&sm.rec[warp][src][2 * sub]) = v;
      }
    }
    __syncwarp();
  }
  if (want) {
    slot[SL_OUT] = keep_out;
    float px, py, pz;
    slot_point(slot, px, py, pz);
    double cx, cy, cz;
    cross_vec(a.extR, a.extT, px, py, pz, cx, cy, cz);
    slot[SL_SPP] = spp_of(load_head(slot), cx, cy, cz, sm.Ptt, sm.Ppp);
  }
}

// Cold: first contact of a lane with its point — the raw point and the body covariance into the slot.
__device__ LIO_COLD void lio_cold_point(const float *__restrict__ pts, const double *__restrict__ pre_base, int pre_stride, int i, double *slot) {
  const float px = pts[3 * (size_t)i], py = pts[3 * (size_t)i + 1], pz = pts[3 * (size_t)i + 2];
  *reinterpret_cast<float2 *>(slot + SL_PT) = make_float2(px, py);
  *reinterpret_cast<float2 *>(slot + SL_ROW + 8) = make_float2(0.f, pz);
  *reinterpret_cast<int2 *>(slot + SL_OUT) = make_int2(-1, -1);
  const size_t ns = (size_t)pre_stride;
  const double *__restrict__ pre = pre_base + i;
  double2 *bc2 = reinterpret_cast<double2 *>(slot + SL_BC);
  bc2[0] = make_double2(pre[3 * ns], pre[4 * ns]);
  bc2[1] = make_double2(pre[5 * ns], pre[6 * ns]);
  bc2[2] = make_double2(pre[7 * ns], pre[8 * ns]);
  reinterpret_cast<int *>(slot + SL_META)[1] = -1;  // no cached R_inv
}

// Cold (once per point and matched plane): R_inv = 1 / (0.001 + sigma_l + n^T var n) with the PRIOR pose (:425-449):
// point_world = Rp p_imu + tp, var = (Rp extR) body_cov (Rp extR)^T  =>  n^T var n = m^T body_cov m, m = Mp^T n.
// Iteration-invariant, cached in the slot together with the plane it belongs to.
__device__ LIO_COLD double lio_cold_wgt(LioSmem &sm, int warp, int lane, const double *__restrict__ q, int plane_idx) {
  double *slot = &sm.rec[warp][lane][0];
  float px, py, pz;
  slot_point(slot, px, py, pz);
  double pi0, pi1, pi2;
  p_imu(sm.cold.extR, sm.cold.extT, px, py, pz, pi0, pi1, pi2);
  const RecHead h = load_head(q);
  const double w0 = sm.Rp[0] * pi0 + sm.Rp[1] * pi1 + sm.Rp[2] * pi2 + sm.tp[0];
  const double w1 = sm.Rp[3] * pi0 + sm.Rp[4] * pi1 + sm.Rp[5] * pi2 + sm.tp[1];
  const double w2 = sm.Rp[6] * pi0 + sm.Rp[7] * pi1 + sm.Rp[8] * pi2 + sm.tp[2];
  const double sigma_l = sigma_plane(q, h.c0 - w0, h.c1 - w1, h.c2 - w2);
  double p0, p1, p2;
  rot_t_n(sm.Mp, h, p0, p1, p2);
  const double wgt = 1.0 / (0.001 + sigma_l + quad_bc(slot + SL_BC, p0, p1, p2));
  slot[SL_WGT] = wgt;
  reinterpret_cast<int *>(slot + SL_META)[1] = plane_idx;
  return wgt;
}
#define LIO_PHASE_FENCE() asm volatile("" ::: "memory")  // keeps the next phase's shared-memory loads from being hoisted (register pressure)

// Kernel start: the slice of the kernel arguments the cold paths read, into shared memory.
__device__ __forceinline__ void lio_init_cold(LioSmem &sm, const LioKernelArgs &a) {
  if (threadIdx.x == 0) {
    LioCold &c = sm.cold;
    c.recs = a.recs, c.slots = a.slots, c.hash_mask = a.hash_mask, c.voxel_size_f = a.voxel_size_f, c.sigma_num = a.sigma_num;
    c.voxel_size = a.voxel_size, c.inv_voxel_size = a.inv_voxel_size, c.inv_voxel_exact = a.inv_voxel_exact, c.stage_mode = a.stage_mode;
    for (int k = 0; k < 9; k++) c.extR[k] = a.extR[k];
    for (int k = 0; k < 3; k++) c.extT[k] = a.extT[k];
  }
}

// Residual / Jacobian build over the points [lo, hi) of this rank's shard (indices local to the shard), accumulated into
// the calling warp's 8x8 tensor-core block (D0, D1) and matched-point count. The CTA walks its block in tiles of
// LIO_THREADS points; with a single tile (the resident case) a lane keeps its point, its slot and `lc` for the whole update.
// write_out: store the per-point outputs (match_plane / dis_to_plane / normal_plane) of this pass to global memory; the
// persistent kernel defers that to its last iteration when the slice is resident (lc.out_* carry the values).
__device__ __forceinline__ void lio_process_range(const LioKernelArgs &a, LioSmem &sm, int lo, int hi, double &D0, double &D1, int &cnt,
                                                  LaneCache &lc, bool init_normal, bool write_out) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double *const slot = &sm.rec[warp][lane][0];
  const bool resident = (hi - lo <= LIO_THREADS);
  for (int base = lo; base < hi; base += LIO_THREADS) {
    const int li = base + tid;
    const bool valid = li < hi;
    const int i = a.begin + li;
    if (!resident) lane_cache_reset(lc);  // several tiles share the lanes: nothing stays resident
    double pw[3] = {0, 0, 0};
    float loc[3] = {0, 0, 0};
    uint32_t first = 0, count = 0;
    bool found = false;

    // ---- phase 1: transform, voxel key, home voxel (cached or probed)
    if (valid) {
      if (!lc.have_pt) {
        lio_cold_point(a.pts, a.pre, a.pre_stride, i, slot);
        lc.have_pt = true;
      }
      float px, py, pz;
      slot_point(slot, px, py, pz);
      double pi0, pi1, pi2;
      p_imu(a.extR, a.extT, px, py, pz, pi0, pi1, pi2);
      pw[0] = (double)(float)__dadd_rn(dot3_rn(sm.R[0], sm.R[1], sm.R[2], pi0, pi1, pi2), sm.t[0]);
      pw[1] = (double)(float)__dadd_rn(dot3_rn(sm.R[3], sm.R[4], sm.R[5], pi0, pi1, pi2), sm.t[1]);
      pw[2] = (double)(float)__dadd_rn(dot3_rn(sm.R[6], sm.R[7], sm.R[8], pi0, pi1, pi2), sm.t[2]);
      // voxel key (voxel_map.cpp:665-671): float quotient, "-1 if negative", truncate. When 1/voxel_size is exact (a power
      // of two: 0.5, 2.0, ...) the multiply gives the bit-identical quotient without the slow fp64 division.
      bool finite = true;
#pragma unroll
      for (int j = 0; j < 3; j++) {
        loc[j] = voxel_coord(pw[j], a.voxel_size, a.inv_voxel_size, a.inv_voxel_exact);
        finite = finite && (fabsf(loc[j]) < 3.0e6f);
      }
      const long long k0 = (long long)loc[0], k1 = (long long)loc[1], k2 = (long long)loc[2];
      const bool inr = finite && key_in_range(k0, k1, k2);
      const unsigned long long pkey = inr ? pack_key(k0, k1, k2) : ESIKF_KEY_EMPTY;
      const ulonglong2 km = *reinterpret_cast<const ulonglong2 *>(slot + SL_KEY);  // {key, {count, wgt_idx}}
      if (inr && lc.key_valid && pkey == km.x) {
        // the voxel of the previous iteration: no hash probe
        count = (uint32_t)(km.y & 0xffffffffull);
        found = (count != LIO_ABSENT);
        if (!found) count = 0;
        first = (uint32_t)(lc.staged_idx >= 0 ? lc.staged_idx : 0);
      } else {
        found = inr && probe(a.slots, a.hash_mask, k0, k1, k2, first, count);
        if (inr) {
          *reinterpret_cast<unsigned long long *>(slot + SL_KEY) = pkey;
          reinterpret_cast<uint32_t *>(slot + SL_META)[0] = found ? count : LIO_ABSENT;
          lc.key_valid = true;
          if (!(found && count > 0)) lc.staged_idx = -1;
        } else {
          lc.key_valid = false, lc.staged_idx = -1;
        }
      }
    }
    // ---- phase 2: bring the first candidate record of the (new) voxel into the lane's slot
    {
      const int cand0 = (valid && found && count > 0) ? (int)first : -1;
      const bool want = cand0 >= 0 && cand0 != lc.staged_idx;
      const unsigned wmask = __ballot_sync(0xffffffffu, want);
      if (wmask) {
        lio_cold_stage(sm, warp, lane, want, cand0, wmask, lc.mphase);
        if (a.stage_mode == 0) lc.mphase ^= 1u;
        if (want) lc.staged_idx = cand0;
      }
    }

    LIO_PHASE_FENCE();
    // ---- phase 3: association. Resident record first (hot path), then the extras of sub-divided voxels / neighbour voxel.
    int best_idx = -1;
    float best_dis = 0.f;
    const bool have0 = valid && found && count > 0;
    bool pass0 = false;
    double sigma0 = 0.0;
    float dis0 = 0.f, dtp0 = 0.f;
    if (have0) {
      // nothing of this block stays live past it but the verdict: the Jacobian phase re-reads the slot (registers)
      const RecHead h0 = load_head(slot);
      const Gate1 g = gate_range(h0, pw);
      if (g.pass) {
        double m0, m1, m2;
        rot_t_n(sm.R, h0, m0, m1, m2);
        const double2 sw = *reinterpret_cast<const double2 *>(slot + SL_SPP);  // {spp, wgt}
        sigma0 = sigma_plane(slot, g.e0, g.e1, g.e2) + quad_bc(slot + SL_BC, m0, m1, m2) + sw.x;
        if ((double)g.dis_to_plane < a.sigma_num * sqrt(sigma0)) pass0 = true, dis0 = (float)g.sd, dtp0 = g.dis_to_plane;
      }
      if (pass0 && count == 1) best_idx = (int)first, best_dis = dis0;
    }
    const bool pend1 = have0 && count > 1;
    const bool need_nb = valid && found && !pend1 && best_idx < 0;  // for pend1 lanes: decided after their extras
    if (__any_sync(0xffffffffu, pend1 || need_nb)) {  // cold: narrow arguments, everything else comes from shared memory
      const AssocOut ao = lio_cold_assoc(sm, warp, lane, (pend1 ? 1u : 0u) | ((valid && found) ? 2u : 0u) | (pass0 ? 4u : 0u), (float)pw[0], (float)pw[1], (float)pw[2],
                                         first, count, sigma0, dis0, dtp0);
      best_idx = ao.idx, best_dis = ao.dis;
    }
    LIO_PHASE_FENCE();

    // ---- phase 4: Jacobian / measurement-noise loop (voxel_map.cpp:414-458) for matched points
    const bool matched = best_idx >= 0;
    double row0 = 0, row1 = 0, row2 = 0, rn0 = 0, rn1 = 0, rn2 = 0, rz = 0, wgt = 0;
    if (matched) {
      const bool hot = have0 && best_idx == (int)first;
      const double *__restrict__ q = hot ? slot : reinterpret_cast<const double *>(a.recs + best_idx);
      double m0, m1, m2;
      {
        const double2 *__restrict__ q2 = reinterpret_cast<const double2 *>(q);
        const double2 a1 = q2[1], a2 = q2[2];  // c2 n0 | n1 n2
        rn0 = a1.y, rn1 = a2.x, rn2 = a2.y;
        m0 = sm.R[0] * rn0 + sm.R[3] * rn1 + sm.R[6] * rn2, m1 = sm.R[1] * rn0 + sm.R[4] * rn1 + sm.R[7] * rn2, m2 = sm.R[2] * rn0 + sm.R[5] * rn1 + sm.R[8] * rn2;
      }
      const double2 sw = *reinterpret_cast<const double2 *>(slot + SL_SPP);  // {spp, wgt}
      wgt = (reinterpret_cast<const int *>(slot + SL_META)[1] == best_idx) ? sw.y : lio_cold_wgt(sm, warp, lane, q, best_idx);
      float px, py, pz;
      slot_point(slot, px, py, pz);
      double pi0, pi1, pi2;
      p_imu(a.extR, a.extT, px, py, pz, pi0, pi1, pi2);
      // A = [p_imu]x R^T n with the CURRENT rotation (:453)
      row0 = -pi2 * m1 + pi1 * m2;
      row1 = pi2 * m0 - pi0 * m2;
      row2 = -pi1 * m0 + pi0 * m1;
      rz = -(double)best_dis;  // meas_vec (:457)
    }
    if (valid) {
      lc.out_valid = true;
      // ptpl_list_ membership of this iteration; pv.normal = plane.normal_ (:744) is sticky across iterations
      int2 *out = reinterpret_cast<int2 *>(slot + SL_OUT);
      const int prev_normal = out->y;
      const int normal_now = matched ? best_idx : (init_normal ? -1 : prev_normal);
      *out = make_int2(best_idx, normal_now);
      if (write_out || !resident) {
        a.match_plane[i] = best_idx;
        a.dis_to_plane[i] = matched ? best_dis : 0.f;  // PointToPlane::dis_to_plane_ of this iteration (0 when unmatched)
        if (matched) a.normal_plane[i] = best_idx;
        else if (init_normal) a.normal_plane[i] = -1;
      }
    }
    cnt += __popc(__ballot_sync(0xffffffffu, matched));

    LIO_PHASE_FENCE();
    // ---- phase 5: stage the 32 rows of this warp and contract them on the fp64 tensor path
    {
      double2 *dst = reinterpret_cast<double2 *>(slot + SL_ROW);
      dst[0] = make_double2(row0, row1);
      dst[1] = make_double2(row2, rn0);
      dst[2] = make_double2(rn1, rn2);
      dst[3] = make_double2(rz, wgt);
      reinterpret_cast<float *>(slot + SL_ROW + 8)[0] = matched ? best_dis : 0.f;  // signed; the contraction takes |.|
    }
    __syncwarp();
    {
      const int g = lane >> 2, t = lane & 3;
      double E0 = 0.0, E1 = 0.0;  // second accumulator pair: two independent DMMA chains per tile
#pragma unroll
      for (int s = 0; s < 8; s++) {
        const double *r = &sm.rec[warp][4 * s + t][SL_ROW];
        const double wv = r[7];
        const double v = (g == 7) ? ((wv != 0.0) ? 1.0 : 0.0) : r[g];  // a_7 = 1 for matched rows (R_inv > 0), else 0
        const double b = (g == 7) ? (double)fabsf(reinterpret_cast<const float *>(r + 8)[0]) : wv * v;
        if (s & 1) dmma_m8n8k4(E0, E1, v, b);
        else dmma_m8n8k4(D0, D1, v, b);
      }
      D0 += E0, D1 += E1;
    }
    __syncwarp();
  }
}

// Per-point outputs of a resident slice, written once after the last iteration of the persistent kernel.
__device__ __forceinline__ void lio_write_outputs(const LioKernelArgs &a, const LioSmem &sm, int lo, int hi, const LaneCache &lc) {
  const int li = lo + threadIdx.x;
  if (li < hi && hi - lo <= LIO_THREADS && lc.out_valid) {
    const int i = a.begin + li;
    const double *slot = &sm.rec[threadIdx.x >> 5][threadIdx.x & 31][0];
    const int2 out = *reinterpret_cast<const int2 *>(slot + SL_OUT);
    a.match_plane[i] = out.x;
    a.dis_to_plane[i] = reinterpret_cast<const float *>(slot + SL_ROW + 8)[0];
    a.normal_plane[i] = out.y;
  }
}

// Contiguous slices of the shard per block in whole warps (32-point chunks), spread as evenly as the chunk count allows:
// every SM of the grid takes part (100 k points = 3125 chunks = 21 or 22 warps on each of 148 SMs).
__device__ __forceinline__ void lio_block_range(int count, int &lo, int &hi) {
  const int chunks = (count + 31) >> 5, g = (int)gridDim.x, b = (int)blockIdx.x;
  const int q = chunks / g, r = chunks % g;
  const int first = b * q + (b < r ? b : r), mine = q + (b < r ? 1 : 0);
  lo = first * 32;
  hi = lo + mine * 32;
  if (lo > count) lo = count;
  if (hi > count) hi = count;
}

__device__ __forceinline__ void lio_init_barriers(LioSmem &sm) {
  if (threadIdx.x < LIO_WARPS) mbar_init(&sm.mbar[threadIdx.x], 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
}

__global__ void __launch_bounds__(LIO_THREADS, 1) lio_residual_kernel(const LioKernelArgs a) {
  if (a.ctrl->stop) return;  // EKF_stop_flg: remaining iterations of the unrolled loop do nothing
  extern __shared__ __align__(128) unsigned char smem_raw[];
  LioSmem &sm = *reinterpret_cast<LioSmem *>(smem_raw);
  lio_init_cold(sm, a);
  lio_init_barriers(sm);
  lio_prior_consts(sm, a);
  lio_cov_consts(sm, a.state + S_COV);
  lio_pose_consts(sm, a.state);
  __syncthreads();
  double D0 = 0.0, D1 = 0.0;  // this lane's two entries of the warp's 8x8 block
  int cnt = 0;
  int lo, hi;
  lio_block_range(a.count, lo, hi);
  LaneCache lc;
  lane_cache_init(lc);
  lio_process_range(a, sm, lo, hi, D0, D1, cnt, lc, a.init_normal != 0, true);
  reduce_info<LIO_WARPS, 6>(sm.red, D0, D1, (double)cnt, a.partials, a.partial_stride, a.info, a.ctrl);
}

}  // namespace esikf
