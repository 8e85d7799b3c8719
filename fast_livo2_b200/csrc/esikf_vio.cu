// VIO kernels of the B200 ESIKF update (sm_100a).
//
//   vio_patch_kernel      : one (level, iteration) of VIOManager::updateState's per-patch loop (reference src/vio.cpp:1556-1634):
//                           projection, bilinear taps on the level-0 image at stride 2^(level+search_level), 64 photometric
//                           residuals and 1x7 Jacobian rows per patch, fused with the H^T H / H^T z / sum(res^2) reduction
//                           (:1660-1662). H_sub (128k x 7 doubles per iteration in the reference) is never materialised.
//   image_patch_kernel    : batched getImagePatch (:203-225)
//   warp_matrix_kernel    : batched getWarpMatrixAffineHomography + getBestSearchLevel (:252-273, 320-331, 701-714)
//   warp_affine_kernel    : batched warpAffine over all pyramid levels (:292-318, 739-742)
//
// Mapping: one warp per visual patch, two pixels per lane. The 64 rows [JdR Jdt cur res] of a patch are staged in shared
// memory and contracted with 16 fp64 tensor-core steps (mma.sync.m8n8k4.f64); per-warp 8x8 blocks are combined in a fixed
// order so the error-gated accept / rollback decision is reproducible.
#include "esikf_dev.cuh"

namespace esikf {

#define VIO_THREADS 512  // 16 warps, one CTA per SM
#define VIO_WARPS (VIO_THREADS / 32)

struct CamDev {
  int model, width, height;
  double fx, fy, cx, cy;
  double d[5];
};

// vk::PinholeCamera::world2cam / vk::EquidistantCamera::world2cam (vikit, unpinned; restated from its published algorithm)
__device__ __forceinline__ void world2cam(const CamDev &cam, double X, double Y, double Z, double &u, double &v) {
  double x = X / Z, y = Y / Z;
  if (cam.model == 0) {
    if (!(fabs(cam.d[0]) > 0.0000001)) {
      u = cam.fx * x + cam.cx;
      v = cam.fy * y + cam.cy;
    } else {
      double r2 = x * x + y * y, r4 = r2 * r2, r6 = r4 * r2;
      double a1 = 2 * x * y, a2 = r2 + 2 * x * x, a3 = r2 + 2 * y * y;
      double cdist = 1 + cam.d[0] * r2 + cam.d[1] * r4 + cam.d[4] * r6;
      double xd = x * cdist + cam.d[2] * a1 + cam.d[3] * a2;
      double yd = y * cdist + cam.d[2] * a3 + cam.d[3] * a1;
      u = xd * cam.fx + cam.cx;
      v = yd * cam.fy + cam.cy;
    }
  } else {
    double r = sqrt(x * x + y * y);
    double theta = atan(r);
    double t2 = theta * theta, t4 = t2 * t2, t6 = t4 * t2, t8 = t4 * t4;
    double theta_d = theta * (1 + cam.d[0] * t2 + cam.d[1] * t4 + cam.d[2] * t6 + cam.d[3] * t8);
    double scaling = (r > 1e-8) ? theta_d / r : 1.0;
    u = cam.fx * x * scaling + cam.cx;
    v = cam.fy * y * scaling + cam.cy;
  }
}
// cam2world -> unit bearing (distorted pinhole: 5 fixed-point iterations as cv::undistortPoints)
__device__ __forceinline__ void cam2world(const CamDev &cam, double u, double v, double f[3]) {
  double x0 = (u - cam.cx) / cam.fx, y0 = (v - cam.cy) / cam.fy;
  double x = x0, y = y0;
  if (cam.model == 0) {
    if (fabs(cam.d[0]) > 0.0000001) {
      for (int it = 0; it < 5; it++) {
        double r2 = x * x + y * y;
        double icdist = 1.0 / (1 + ((cam.d[4] * r2 + cam.d[1]) * r2 + cam.d[0]) * r2);
        double dx = 2 * cam.d[2] * x * y + cam.d[3] * (r2 + 2 * x * x);
        double dy = cam.d[2] * (r2 + 2 * y * y) + 2 * cam.d[3] * x * y;
        x = (x0 - dx) * icdist;
        y = (y0 - dy) * icdist;
      }
    }
  } else {
    double theta_d = sqrt(x0 * x0 + y0 * y0);
    if (theta_d > 1e-8) {
      double theta = theta_d;
      for (int it = 0; it < 10; it++) {
        double t2 = theta * theta, t4 = t2 * t2, t6 = t4 * t2, t8 = t4 * t4;
        theta = theta_d / (1 + cam.d[0] * t2 + cam.d[1] * t4 + cam.d[2] * t6 + cam.d[3] * t8);
      }
      double scaling = tan(theta) / theta_d;
      x = x0 * scaling;
      y = y0 * scaling;
    }
  }
  double n = sqrt(x * x + y * y + 1.0);
  f[0] = x / n, f[1] = y / n, f[2] = 1.0 / n;
}

struct VioKernelArgs {
  const uint8_t *img;
  CamDev cam;
  const double *pos;           // [n_total][3]
  const float *warp_patch;     // [n_total][levels*64]
  const int32_t *search_levels;
  const double *inv_expo_list;
  int begin, count;            // this rank's shard of the patches
  int levels, level, slot_iter, exposure_en;
  const double *state;         // current iterate
  double Rci[9], Pci[3], Jdp_dR[9];
  float *errors;               // [n_total]
  double *partials;
  int partial_stride;
  double *info;
  Ctrl *ctrl;
};

// raw img.data + offset reads of the reference, with 0 outside the buffer (the reference would read out of bounds there)
__device__ __forceinline__ float tap(const uint8_t *__restrict__ img, long idx, long npix) {
  return (idx >= 0 && idx < npix) ? (float)__ldg(img + idx) : 0.0f;
}
// w_tl*a + w_tr*b + w_bl*c + w_br*d in float, left to right, no FMA contraction (vio.cpp:1600-1620)
__device__ __forceinline__ float bil(float wtl, float wtr, float wbl, float wbr, float a, float b, float c, float d) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(wtl, a), __fmul_rn(wtr, b)), __fmul_rn(wbl, c)), __fmul_rn(wbr, d));
}

// What a warp keeps about one of ITS patches across the iterations of a persistent update: the iteration-invariant inputs,
// the 11 x 11 strided tap footprint of the level-0 image (re-staged only when the integer tap base or the stride moves —
// sub-pixel motion between iterations leaves it in place) and the 64 reference-patch values of the current pyramid level.
// With it a steady-state iteration of a patch touches no global memory at all.
#define VIO_KMAX 2  // cached patches per warp (2 x 16 warps x 148 SMs = 4.7 k patches resident)
struct VioPatchCache {
  double X, Y, Z, inv_ref_expo;
  long long tile_base0;  // linear index of tile (0,0) in the image the taps were staged from
  int search_level, tile_scale, pv_level, have;
  float taps[128];       // 11 x 11 strided image taps of the patch footprint (level-0 image, stride 2^pyramid_level)
  float pv[64];          // warp_patch of the level being processed
};

// Tap footprints through the TMA unit (tuning flag ESIKF_TUNE_VIO_TMA): one tiled tensor map of the u8 image per tap
// stride s = 1, 2, 4, 8 — box {W_s bytes, 11 s rows} traversed with elementStrides {1, s} (TMA cannot stride the
// innermost dimension), i.e. 11 image rows of W_s contiguous bytes land in shared memory with ONE instruction issued by
// one lane; the 11 x 11 taps are then picked out at stride s. The box must START on a 16-byte boundary of the innermost
// dimension (measured: tools/tma_probe.cu — an unaligned x coordinate raises an illegal-instruction fault on sm_100,
// profiles/tma_probe_r02.txt), so the start pixel is rounded down to a multiple of 16 and W_s = 16 ceil((16 + 10 s) / 16)
// covers the worst offset: 32, 48, 64, 96 bytes. Footprints that leave the image (the reference's raw linear-index reads
// wrap to the neighbouring row there, TMA would zero-fill) and strides 16 / 32 (elementStrides <= 8) keep the per-lane loads.
#define VIO_TMA_MAXLVL 3
#define VIO_TMA_INNER(l) (16u * ((16u + (10u << (l)) + 15u) / 16u))
#define VIO_TMA_TILE_BYTES (11 * 96 + 96)
struct VioTma {
  alignas(64) unsigned char map[VIO_TMA_MAXLVL + 1][128];  // CUtensorMap per level (opaque 128-byte descriptors)
  int enabled;
};

struct __align__(128) VioSmem {
  double rows[VIO_WARPS][64][8];  // first: double4 stores need 32-byte alignment
  alignas(128) unsigned char tile[VIO_WARPS][VIO_TMA_TILE_BYTES];  // TMA landing area of a warp's footprint (u8 rows)
  unsigned long long tma_bar[VIO_WARPS];
  VioPatchCache cache[VIO_WARPS][VIO_KMAX];
  float grid[VIO_WARPS][104];     // 10 x 10 bilinear values: patch pixels plus a one-pixel ring for the central differences
  double Rcw[9], Pcw[3];
  double inv_expo;
  ReduceSmem<VIO_WARPS> red;
};

// Per-iteration constants of updateState (vio.cpp:1540-1544): Rcw, Pcw, inv_expo_time out of the packed state `st` (global
// memory in the per-iteration kernels, the CTA's resident copy in the persistent one).
__device__ __forceinline__ void vio_pose_consts(VioSmem &sm, const VioKernelArgs &a, const double *st) {
  const int tid = threadIdx.x;
  if (tid < 9) {
    // Rcw = Rci * Rwi^T  (vio.cpp:1542)
    const int r = tid / 3, c = tid % 3;
    double s = 0;
    for (int k = 0; k < 3; k++) s += a.Rci[r * 3 + k] * st[S_R + c * 3 + k];
    sm.Rcw[tid] = s;
  }
  if (tid == 0) sm.inv_expo = st[S_EXPO];
  __syncthreads();
  if (tid < 3) {
    // Pcw = -Rci Rwi^T Pwi + Pci  (:1543)
    double s = 0;
    for (int k = 0; k < 3; k++) s += sm.Rcw[tid * 3 + k] * st[S_P + k];
    sm.Pcw[tid] = -s + a.Pci[tid];
  }
  __syncthreads();
}

// Integer tap base and bilinear weights of a patch centred at (pcu, pcv) with tap stride 2^pyramid_level (vio.cpp:206-215,
// 1580-1589) — float, via double (1.0 - subpix). Divisions by the stride are multiplications with its exact
// reciprocal: x / 2^k and x * 2^-k are the same real number, so the rounded quotient is the same bit for bit.
struct Bilinear {
  int u_ref_i, v_ref_i;
  float w_tl, w_tr, w_bl, w_br;
};
__device__ __forceinline__ Bilinear bilinear_setup(double pcu, double pcv, int pyramid_level) {
  const int scale = 1 << pyramid_level;
  // 2^-pyramid_level assembled from its exponent bits — the value 1.0f / (float)scale has
  const float inv_scale = __int_as_float((127 - pyramid_level) << 23);
  const double inv_scale_d = __longlong_as_double((long long)(1023 - pyramid_level) << 52);
  const float u_ref = (float)pcu, v_ref = (float)pcv;
  Bilinear b;
  b.u_ref_i = (int)(floorf((float)(pcu * inv_scale_d)) * scale);
  b.v_ref_i = (int)(floorf((float)(pcv * inv_scale_d)) * scale);
  const float subpix_u = __fmul_rn(u_ref - (float)b.u_ref_i, inv_scale);
  const float subpix_v = __fmul_rn(v_ref - (float)b.v_ref_i, inv_scale);
  b.w_tl = (float)((1.0 - subpix_u) * (1.0 - subpix_v));
  b.w_tr = (float)(subpix_u * (1.0 - subpix_v));
  b.w_bl = (float)((1.0 - subpix_u) * subpix_v);
  b.w_br = subpix_u * subpix_v;
  return b;
}

__device__ __forceinline__ void vio_cache_reset(VioSmem &sm) {
  for (int t = threadIdx.x; t < VIO_WARPS * VIO_KMAX; t += blockDim.x) {
    VioPatchCache &c = sm.cache[t / VIO_KMAX][t % VIO_KMAX];
    c.have = 0, c.pv_level = -1, c.tile_scale = 0, c.tile_base0 = 0;
  }
}

// Photometric residual / Jacobian build of the patches [lo, hi) of this rank's shard at pyramid level `level`.
// Patch lo + warp + 16 k belongs to (warp, k). cached: the CTA's patches fit the per-warp cache (k < VIO_KMAX) and the
// caller keeps `sm.cache` alive between calls (persistent kernel); otherwise slot 0 is plain scratch, refilled every time.
__device__ __forceinline__ void vio_process_range(const VioKernelArgs &a, VioSmem &sm, int level, int lo, int hi, double &D0, double &D1,
                                                  double &n_meas, bool cached, const VioTma *tma = nullptr, unsigned *tma_phase = nullptr) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long npix = (long)a.cam.width * a.cam.height;
  const int width = a.cam.width;
  const double inv_expo = sm.inv_expo;
  float *const sG = sm.grid[warp];
  int k = 0;
  for (int lp = lo + warp; lp < hi; lp += VIO_WARPS, k++) {
    const int i = a.begin + lp;
    VioPatchCache &c = sm.cache[warp][cached ? k : 0];
    const bool fill = !cached || !c.have;  // decisions on the shared slot are read first, acted on after a warp barrier
    __syncwarp();
    if (fill) {
      if (lane == 0) {
        c.search_level = a.search_levels[i];
        c.X = a.pos[3 * (size_t)i], c.Y = a.pos[3 * (size_t)i + 1], c.Z = a.pos[3 * (size_t)i + 2];
        c.inv_ref_expo = a.inv_expo_list[i];
        c.have = 1, c.pv_level = -1, c.tile_scale = 0;
      }
      __syncwarp();
    }
    const int search_level = c.search_level;
    const double X = c.X, Y = c.Y, Z = c.Z, inv_ref_expo = c.inv_ref_expo;
    const int pyramid_level = level + search_level;
    const int scale = 1 << pyramid_level;
    const float inv_scale = __int_as_float((127 - pyramid_level) << 23);  // 2^-pyramid_level, the value 1.0f / (float)scale has
    const double pf0 = sm.Rcw[0] * X + sm.Rcw[1] * Y + sm.Rcw[2] * Z + sm.Pcw[0];
    const double pf1 = sm.Rcw[3] * X + sm.Rcw[4] * Y + sm.Rcw[5] * Z + sm.Pcw[1];
    const double pf2 = sm.Rcw[6] * X + sm.Rcw[7] * Y + sm.Rcw[8] * Z + sm.Pcw[2];
    double pcu, pcv;
    world2cam(a.cam, pf0, pf1, pf2, pcu, pcv);
    const Bilinear bw = bilinear_setup(pcu, pcv, pyramid_level);
    const int u_ref_i = bw.u_ref_i, v_ref_i = bw.v_ref_i;

    // the 11 x 11 tap footprint: tile (r, c) <-> image linear index base0 + r*scale*width + c*scale, where tile (1,1) is the
    // top-left tap of patch pixel (0,0) (:1597). Staged only when the footprint moved.
    // The loads are issued here and consumed after the Jacobian constants below (their latency hides behind that math).
    float tv[4] = {0.f, 0.f, 0.f, 0.f};
    bool restage, by_tma = false;
    {
      const long long base0 = (long long)(v_ref_i - 5 * scale) * width + (u_ref_i - 5 * scale);
      const bool repv = (c.pv_level != level);
      restage = (c.tile_scale != scale || c.tile_base0 != base0);
      __syncwarp();
      if (restage) {
        const int x0 = u_ref_i - 5 * scale, y0 = v_ref_i - 5 * scale;
        by_tma = tma && pyramid_level <= VIO_TMA_MAXLVL && x0 >= 0 && y0 >= 0 && x0 + 10 * scale < width && y0 + 10 * scale < a.cam.height;
        if (by_tma) {
          if (lane == 0) {
            fence_proxy_async_smem();  // the landing area was last read through the generic proxy
            mbar_arrive_expect_tx(&sm.tma_bar[warp], 11u * VIO_TMA_INNER(pyramid_level));
            tma_load_2d(sm.tile[warp], tma->map[pyramid_level], x0 & ~15, y0, &sm.tma_bar[warp]);
          }
        } else {
          const long sw = (long)scale * width;
#pragma unroll
          for (int q = 0; q < 4; q++) {
            const int t = lane + 32 * q;
            if (t < 121) {
              const int r = t / 11, cc = t - 11 * r;
              tv[q] = tap(a.img, (long)base0 + r * sw + (long)cc * scale, npix);
            }
          }
        }
        if (lane == 0) c.tile_scale = scale, c.tile_base0 = base0;
      }
      if (repv) {
        const float2 v = *reinterpret_cast<const float2 *>(a.warp_patch + (size_t)i * 64 * a.levels + 64 * level + 2 * lane);
        *reinterpret_cast<float2 *>(&c.pv[2 * lane]) = v;
        if (lane == 0) c.pv_level = level;
      }
    }
    // computeProjectionJacobian (:189-201) and the per-patch 2x3 maps so that per pixel JdR = [du dv] WR, Jdt = [du dv] WT (:1611-1617):
    //   Jimg = [du dv] * inv_expo * inv_scale ; Jdphi = Jimg Jdpi [pf]x ; Jdp = -Jimg Jdpi ; JdR = Jdphi Rci + Jdp Jdp_dR ; Jdt = Jdp Rcw
    const double z_inv = 1. / pf2, z_inv_2 = z_inv * z_inv;
    const double J00 = a.cam.fx * z_inv, J02 = -a.cam.fx * pf0 * z_inv_2, J11 = a.cam.fy * z_inv, J12 = -a.cam.fy * pf1 * z_inv_2;
    const double sc = inv_expo * (double)inv_scale;
    const double Q00 = J02 * (-pf1), Q01 = J00 * (-pf2) + J02 * pf0, Q02 = J00 * pf1;  // Jdpi [pf]x
    const double Q10 = J11 * pf2 + J12 * (-pf1), Q11 = J12 * pf0, Q12 = J11 * (-pf0);
    double WR[2][3], WT[2][3];
#pragma unroll
    for (int cc = 0; cc < 3; cc++) {
      WR[0][cc] = sc * ((Q00 * a.Rci[cc] + Q01 * a.Rci[3 + cc] + Q02 * a.Rci[6 + cc]) - (J00 * a.Jdp_dR[cc] + J02 * a.Jdp_dR[6 + cc]));
      WR[1][cc] = sc * ((Q10 * a.Rci[cc] + Q11 * a.Rci[3 + cc] + Q12 * a.Rci[6 + cc]) - (J11 * a.Jdp_dR[3 + cc] + J12 * a.Jdp_dR[6 + cc]));
      WT[0][cc] = -sc * (J00 * sm.Rcw[cc] + J02 * sm.Rcw[6 + cc]);
      WT[1][cc] = -sc * (J11 * sm.Rcw[3 + cc] + J12 * sm.Rcw[6 + cc]);
    }
    if (restage) {
      if (by_tma) {
        mbar_wait(&sm.tma_bar[warp], *tma_phase & 1u);
        *tma_phase ^= 1u;
        const unsigned inner = VIO_TMA_INNER(pyramid_level);
        const unsigned char *raw = sm.tile[warp] + ((u_ref_i - 5 * scale) & 15);  // the box starts at the 16-byte boundary below the first tap
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int t = lane + 32 * q;
          if (t < 121) {
            const int r = t / 11, cc = t - 11 * r;
            c.taps[t] = (float)raw[r * inner + (unsigned)cc * scale];
          }
        }
      } else {
#pragma unroll
        for (int q = 0; q < 4; q++)
          if (lane + 32 * q < 121) c.taps[lane + 32 * q] = tv[q];
      }
    }
    __syncwarp();
    const float *const sT = c.taps;
    // bilinear value grid: G(a,b) = cur_value of patch pixel (a-1, b-1), a,b in 0..9 (same float op order as :1619-1620)
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int g = lane + 32 * q;
      if (g < 100) {
        const int ga = g / 10, gb = g - 10 * ga;
        const float *t0 = sT + ga * 11 + gb;
        sG[g] = bil(bw.w_tl, bw.w_tr, bw.w_bl, bw.w_br, t0[0], t0[1], t0[11], t0[12]);
      }
    }
    __syncwarp();
    const float2 Pv = *reinterpret_cast<const float2 *>(&c.pv[2 * lane]);
#pragma unroll
    for (int q = 0; q < 2; q++) {
      const int pix = 2 * lane + q;  // = x*8 + y
      const int x = pix >> 3, y = pix & 7;
      const float *gc = sG + (x + 1) * 10 + (y + 1);
      // du = 0.5f * (cur(x, y+1) - cur(x, y-1)), dv = 0.5f * (cur(x+1, y) - cur(x-1, y))   (:1600-1609)
      const float du = __fmul_rn(0.5f, __fsub_rn(gc[1], gc[-1]));
      const float dv = __fmul_rn(0.5f, __fsub_rn(gc[10], gc[-10]));
      const double cur_value = (double)gc[0];
      const double res = inv_expo * cur_value - inv_ref_expo * (double)(q == 0 ? Pv.x : Pv.y);
      const double ddu = (double)du, ddv = (double)dv;
      double4 *dst = reinterpret_cast<double4 *>(&sm.rows[warp][pix][0]);
      dst[0] = make_double4(ddu * WR[0][0] + ddv * WR[1][0], ddu * WR[0][1] + ddv * WR[1][1], ddu * WR[0][2] + ddv * WR[1][2],
                            ddu * WT[0][0] + ddv * WT[1][0]);
      dst[1] = make_double4(ddu * WT[0][1] + ddv * WT[1][1], ddu * WT[0][2] + ddv * WT[1][2], a.exposure_en ? cur_value : 0.0, res);
    }
    n_meas += 64.0;
    __syncwarp();
    {
      // four independent accumulator pairs: the 16 contraction steps form 4 dependency chains of 4 instead of one of 16
      const int g = lane >> 2, t = lane & 3;
      double A0 = 0.0, A1 = 0.0, B0 = 0.0, B1 = 0.0, C0 = 0.0, C1 = 0.0, E0 = 0.0, E1 = 0.0;
#pragma unroll
      for (int s = 0; s < 16; s += 4) {
        const double v0 = sm.rows[warp][4 * s + t][g], v1 = sm.rows[warp][4 * s + 4 + t][g], v2 = sm.rows[warp][4 * s + 8 + t][g], v3 = sm.rows[warp][4 * s + 12 + t][g];
        dmma_m8n8k4(A0, A1, v0, v0);
        dmma_m8n8k4(B0, B1, v1, v1);
        dmma_m8n8k4(C0, C1, v2, v2);
        dmma_m8n8k4(E0, E1, v3, v3);
      }
      const double p0 = (A0 + B0) + (C0 + E0), p1 = (A1 + B1) + (C1 + E1);  // this patch's 8 x 8 block
      D0 += p0, D1 += p1;
      // patch error (visual_submap->errors[i], :1632) = sum of the 64 squared residuals = element (7, 7) of the patch's block
      // (lane 31 holds it): fp64 sum narrowed to float, no separate reduction
      if (lane == 31) a.errors[i] = (float)p1;
    }
    __syncwarp();
  }
}

__device__ __forceinline__ void vio_block_range(int count, int &lo, int &hi) {
  const int per = (count + gridDim.x - 1) / gridDim.x;
  lo = blockIdx.x * per;
  hi = lo + per < count ? lo + per : count;
  if (lo > count) lo = count;
}

__global__ void __launch_bounds__(VIO_THREADS, 1) vio_patch_kernel(const VioKernelArgs a) {
  if (a.slot_iter > 0 && a.ctrl->level_done) return;  // EKF_end of this level: remaining slots do nothing
  extern __shared__ __align__(128) unsigned char smem_raw[];
  VioSmem &sm = *reinterpret_cast<VioSmem *>(smem_raw);
  vio_pose_consts(sm, a, a.state);
  double D0 = 0.0, D1 = 0.0, n_meas = 0.0;
  int lo, hi;
  vio_block_range(a.count, lo, hi);
  vio_process_range(a, sm, a.level, lo, hi, D0, D1, n_meas, false);
  reduce_info<VIO_WARPS, 7>(sm.red, D0, D1, n_meas, a.partials, a.partial_stride, a.info, a.ctrl);
}


// ---------------------------------------------------------------------------------------------------------------------
// getImagePatch (vio.cpp:203-225), one thread per output pixel.
__global__ void image_patch_kernel(const uint8_t *__restrict__ img, int width, int height, const double *__restrict__ pc, int n, int level,
                                   float *__restrict__ out) {
  int gid = blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= n * 64) return;
  int i = gid >> 6, pix = gid & 63, x = pix >> 3, y = pix & 7;
  const int scale = 1 << level;
  const Bilinear bw = bilinear_setup(pc[2 * i], pc[2 * i + 1], level);
  const long npix = (long)width * height;
  const long b = (long)(bw.v_ref_i - 4 * scale + x * scale) * width + (bw.u_ref_i - 4 * scale) + (long)y * scale;
  const long sw = (long)scale * width;
  out[gid] = bil(bw.w_tl, bw.w_tr, bw.w_bl, bw.w_br, tap(img, b, npix), tap(img, b + scale, npix), tap(img, b + sw, npix), tap(img, b + sw + scale, npix));
}

// getWarpMatrixAffineHomography + getBestSearchLevel for the normal_en branch of retrieveFromVisualSparseMap (vio.cpp:699-715).
__global__ void warp_matrix_kernel(CamDev cam, int n, const double *__restrict__ px_ref, const double *__restrict__ pos_w,
                                   const double *__restrict__ normal_w, const double *__restrict__ T_ref_w, const double *__restrict__ T_cur_w,
                                   double *__restrict__ A_out, int32_t *__restrict__ search_level) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double *Rr = T_ref_w + 12 * (size_t)i, *tr = Rr + 9;
  const double *Rc = T_cur_w, *tc = T_cur_w + 9;
  const double *nw = normal_w + 3 * (size_t)i, *pw = pos_w + 3 * (size_t)i;
  // norm_vec = (R_ref * normal).normalized(); pf = T_ref * pos   (:701-703)
  double nv[3], pf[3];
  for (int r = 0; r < 3; r++) {
    nv[r] = Rr[3 * r] * nw[0] + Rr[3 * r + 1] * nw[1] + Rr[3 * r + 2] * nw[2];
    pf[r] = Rr[3 * r] * pw[0] + Rr[3 * r + 1] * pw[1] + Rr[3 * r + 2] * pw[2] + tr[r];
  }
  double nn = sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]);
  nv[0] /= nn, nv[1] /= nn, nv[2] /= nn;
  // T_cur_ref = T_cur * T_ref^-1 : R = Rc Rr^T, t = tc - R tr   (:710)
  double R[9], t[3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) R[3 * r + c] = Rc[3 * r] * Rr[3 * c] + Rc[3 * r + 1] * Rr[3 * c + 1] + Rc[3 * r + 2] * Rr[3 * c + 2];
  for (int r = 0; r < 3; r++) t[r] = tc[r] - (R[3 * r] * tr[0] + R[3 * r + 1] * tr[1] + R[3 * r + 2] * tr[2]);
  // t_inv = T_cur_ref.inverse().translation() = -R^T t   (:256)
  double ti[3];
  for (int r = 0; r < 3; r++) ti[r] = -(R[r] * t[0] + R[3 + r] * t[1] + R[6 + r] * t[2]);
  // H = R * (n.xyz * I - t_inv n^T)   (:257-258)
  const double ndx = nv[0] * pf[0] + nv[1] * pf[1] + nv[2] * pf[2];
  double Bm[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) Bm[3 * r + c] = ((r == c) ? ndx : 0.0) - ti[r] * nv[c];
  double H[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) H[3 * r + c] = R[3 * r] * Bm[c] + R[3 * r + 1] * Bm[3 + c] + R[3 * r + 2] * Bm[6 + c];
  double fdu[3], fdv[3];
  cam2world(cam, px_ref[2 * i] + 4.0, px_ref[2 * i + 1], fdu);  // level_ref = 0 (:712)
  cam2world(cam, px_ref[2 * i], px_ref[2 * i + 1] + 4.0, fdv);
  double fc[3], fu[3], fv[3];
  for (int r = 0; r < 3; r++) {
    fc[r] = H[3 * r] * pf[0] + H[3 * r + 1] * pf[1] + H[3 * r + 2] * pf[2];
    fu[r] = H[3 * r] * fdu[0] + H[3 * r + 1] * fdu[1] + H[3 * r + 2] * fdu[2];
    fv[r] = H[3 * r] * fdv[0] + H[3 * r + 1] * fdv[1] + H[3 * r + 2] * fdv[2];
  }
  double cu, cv, uu, uv, vu, vv;
  world2cam(cam, fc[0], fc[1], fc[2], cu, cv);
  world2cam(cam, fu[0], fu[1], fu[2], uu, uv);
  world2cam(cam, fv[0], fv[1], fv[2], vu, vv);
  const double A00 = (uu - cu) / 4, A10 = (uv - cv) / 4, A01 = (vu - cu) / 4, A11 = (vv - cv) / 4;
  A_out[4 * i] = A00, A_out[4 * i + 1] = A01, A_out[4 * i + 2] = A10, A_out[4 * i + 3] = A11;
  // getBestSearchLevel(A, 2)   (:320-331)
  int sl = 0;
  double Dt = A00 * A11 - A01 * A10;
  while (Dt > 3.0 && sl < 2) {
    sl += 1;
    Dt *= 0.25;
  }
  search_level[i] = sl;
}

// warpAffine for all pyramid levels (vio.cpp:292-318, 739-742). One thread per output value.
__global__ void warp_affine_kernel(const uint8_t *const *__restrict__ ref_imgs, const int32_t *__restrict__ ref_idx, int cols, int rows, int n,
                                   int levels, const double *__restrict__ A_cur_ref, const double *__restrict__ px_ref,
                                   const int32_t *__restrict__ search_level, float *__restrict__ out) {
  int gid = blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= n * levels * 64) return;
  const int i = gid / (levels * 64), rem = gid % (levels * 64), pyramid_level = rem >> 6, pix = rem & 63, y = pix >> 3, x = pix & 7;
  const double a00 = A_cur_ref[4 * i], a01 = A_cur_ref[4 * i + 1], a10 = A_cur_ref[4 * i + 2], a11 = A_cur_ref[4 * i + 3];
  const double det = a00 * a11 - a01 * a10;
  const double id = 1.0 / det;
  const float A00 = (float)(a11 * id), A01 = (float)(-a01 * id), A10 = (float)(-a10 * id), A11 = (float)(a00 * id);
  if (isnan(A00)) return;  // :297-301 (patch left untouched)
  float pp0 = (float)(x - 4), pp1 = (float)(y - 4);
  const float s1 = (float)(1 << search_level[i]), s2 = (float)(1 << pyramid_level);
  pp0 = __fmul_rn(__fmul_rn(pp0, s1), s2);
  pp1 = __fmul_rn(__fmul_rn(pp1, s1), s2);
  const float px0 = __fadd_rn(__fadd_rn(__fmul_rn(A00, pp0), __fmul_rn(A01, pp1)), (float)px_ref[2 * i]);
  const float px1 = __fadd_rn(__fadd_rn(__fmul_rn(A10, pp0), __fmul_rn(A11, pp1)), (float)px_ref[2 * i + 1]);
  float val = 0.0f;
  // in-frame test of :312 written so that a NaN position (singular A with zero entries: inf * 0) counts as outside; the
  // reference would hand NaN to vk::interpolateMat_8u and read out of bounds
  if (px0 >= 0 && px1 >= 0 && px0 < (float)(cols - 1) && px1 < (float)(rows - 1)) {
    // vk::interpolateMat_8u
    const uint8_t *__restrict__ img = ref_imgs[ref_idx[i]];
    const int xi = (int)floorf(px0), yi = (int)floorf(px1);
    const float sx = px0 - (float)xi, sy = px1 - (float)yi;
    const float w00 = __fmul_rn(1.0f - sx, 1.0f - sy), w01 = __fmul_rn(1.0f - sx, sy), w10 = __fmul_rn(sx, 1.0f - sy);
    const float w11 = __fsub_rn(__fsub_rn(__fsub_rn(1.0f, w00), w01), w10);  // vikit: the last weight is the remainder 1 - w00 - w01 - w10
    const uint8_t *p = img + (long)yi * cols + xi;
    val = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w00, (float)p[0]), __fmul_rn(w01, (float)p[cols])), __fmul_rn(w10, (float)p[1])),
                    __fmul_rn(w11, (float)p[cols + 1]));
  }
  out[gid] = val;
}

// ---------------------------------------------------------------------------------------------------------------------
// Inverse-compositional variant (vio/inverse_composition_en, src/vio.cpp:792-795, 1327-1518): the Jacobian rows come from the
// gradients of each point's REFERENCE image, computed once per pyramid level in the world frame (H_sub_inv) and rotated into
// the current IMU frame every iteration; the residual has no exposure factors and H has 6 columns. It runs inside the
// persistent vio_update_kernel or, per-iteration, as one launch per (level, iteration) like the forward path; the solve is
// the forward one unchanged (with a zero 7th column the 7 x 7 gain elimination reproduces the 6 x 6 one exactly).
struct VioInvArgs {
  const uint8_t *const *ref_imgs;  // registered reference images (Feature::img_)
  const int32_t *ref_idx;          // [n] image of point i
  const double *ref_px;            // [n][2] Feature::px_
  const double *ref_f;             // [n][3] Feature::f_
  const double *ref_R;             // [n][9] Feature::T_f_w_ rotation
  const double *ref_pos;           // [n][3] Feature::pos()
  double *H_sub_inv;               // [n][64][6] rows of the level being processed
  int ref_w, ref_h;
  double fx, fy;
};

// precomputeReferencePatches (:1327-1396) for one point at one level by one warp, two pixels per lane.
__device__ __forceinline__ void vio_inverse_precompute_patch(const VioKernelArgs &a, const VioInvArgs &v, int level, int lp, int lane) {
  const int i = a.begin + lp;
  const int scale = 1 << level;
  const uint8_t *__restrict__ img = v.ref_imgs[v.ref_idx[i]];
  const long npix = (long)v.ref_w * v.ref_h;
  const int width = v.ref_w;
  const double X = a.pos[3 * (size_t)i], Y = a.pos[3 * (size_t)i + 1], Z = a.pos[3 * (size_t)i + 2];
  const double dx = X - v.ref_pos[3 * (size_t)i], dy = Y - v.ref_pos[3 * (size_t)i + 1], dz = Z - v.ref_pos[3 * (size_t)i + 2];
  const double depth = sqrt(dx * dx + dy * dy + dz * dz);
  const double pf0 = v.ref_f[3 * (size_t)i] * depth, pf1 = v.ref_f[3 * (size_t)i + 1] * depth, pf2 = v.ref_f[3 * (size_t)i + 2] * depth;
  const double z_inv = 1. / pf2, z_inv_2 = z_inv * z_inv;
  const double J00 = v.fx * z_inv, J02 = -v.fx * pf0 * z_inv_2, J11 = v.fy * z_inv, J12 = -v.fy * pf1 * z_inv_2;
  const double *R = v.ref_R + 9 * (size_t)i;
  // B = Jdpi * R_ref_w (2 x 3); C = B * [pos]x (2 x 3): per pixel JdR = Jimg C, Jdt = -Jimg B with Jimg = [du dv] / scale
  double B[2][3], Cm[2][3];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    B[0][c] = J00 * R[c] + J02 * R[6 + c];
    B[1][c] = J11 * R[3 + c] + J12 * R[6 + c];
  }
#pragma unroll
  for (int r = 0; r < 2; r++) {
    Cm[r][0] = B[r][1] * Z - B[r][2] * Y;   // B * skew(pos): column 0 = B1 * Z + B2 * (-Y)
    Cm[r][1] = -B[r][0] * Z + B[r][2] * X;
    Cm[r][2] = B[r][0] * Y - B[r][1] * X;
  }
  const Bilinear bw = bilinear_setup(v.ref_px[2 * (size_t)i], v.ref_px[2 * (size_t)i + 1], level);
  const float w_tl = bw.w_tl, w_tr = bw.w_tr, w_bl = bw.w_bl, w_br = bw.w_br;
  const double inv_scale = 1.0 / scale;
  const long sw = (long)scale * width;
#pragma unroll
  for (int k = 0; k < 2; k++) {
    const int pix = 2 * lane + k, x = pix >> 3, y = pix & 7;
    const long b = (long)(bw.v_ref_i + x * scale - 4 * scale) * width + (bw.u_ref_i - 4 * scale) + (long)y * scale;
    const float du = __fmul_rn(0.5f, __fsub_rn(bil(w_tl, w_tr, w_bl, w_br, tap(img, b + scale, npix), tap(img, b + 2 * scale, npix), tap(img, b + sw + scale, npix),
                                                 tap(img, b + sw + 2 * scale, npix)),
                                             bil(w_tl, w_tr, w_bl, w_br, tap(img, b - scale, npix), tap(img, b, npix), tap(img, b + sw - scale, npix), tap(img, b + sw, npix))));
    const float dv = __fmul_rn(0.5f, __fsub_rn(bil(w_tl, w_tr, w_bl, w_br, tap(img, b + sw, npix), tap(img, b + scale + sw, npix), tap(img, b + 2 * sw, npix),
                                                 tap(img, b + 2 * sw + scale, npix)),
                                             bil(w_tl, w_tr, w_bl, w_br, tap(img, b - sw, npix), tap(img, b - sw + scale, npix), tap(img, b, npix), tap(img, b + scale, npix))));
    const double ju = (double)du * inv_scale, jv = (double)dv * inv_scale;
    double *h = v.H_sub_inv + ((size_t)lp * 64 + pix) * 6;
#pragma unroll
    for (int c = 0; c < 3; c++) {
      h[c] = ju * Cm[0][c] + jv * Cm[1][c];
      h[3 + c] = -(ju * B[0][c] + jv * B[1][c]);
    }
  }
}
__global__ void vio_inverse_precompute_kernel(const VioKernelArgs a, const VioInvArgs v, int level) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lp = blockIdx.x * (blockDim.x >> 5) + warp;
  if (lp >= a.count) return;
  vio_inverse_precompute_patch(a, v, level, lp, lane);
}

// Measurement build of updateStateInverse (:1420-1480) over the patches [lo, hi) of this rank's shard at pyramid level
// `level`: residual / rows contracted on the tensor-core path into the same 8 x 8 block layout as the forward kernel (H^T H
// in [0..5][0..5], row / column 6 zero, H^T z in column 7, sum res^2 in [7][7]). `st`: the packed current state, as for
// vio_pose_consts. Shared by the per-iteration kernel and the persistent kernel (bit-identical).
__device__ __forceinline__ void vio_inverse_process_range(const VioKernelArgs &a, const VioInvArgs &v, VioSmem &sm, int level, int lo, int hi, const double *st,
                                                          double &D0, double &D1, double &n_meas) {
  const double *const Rwi = st + S_R, *const Pwi = st + S_P;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int scale = 1 << level;
  const long npix = (long)a.cam.width * a.cam.height;
  const int width = a.cam.width;
  for (int lp = lo + warp; lp < hi; lp += VIO_WARPS) {
    const int i = a.begin + lp;
    const double X = a.pos[3 * (size_t)i], Y = a.pos[3 * (size_t)i + 1], Z = a.pos[3 * (size_t)i + 2];
    const double pf0 = sm.Rcw[0] * X + sm.Rcw[1] * Y + sm.Rcw[2] * Z + sm.Pcw[0];
    const double pf1 = sm.Rcw[3] * X + sm.Rcw[4] * Y + sm.Rcw[5] * Z + sm.Pcw[1];
    const double pf2 = sm.Rcw[6] * X + sm.Rcw[7] * Y + sm.Rcw[8] * Z + sm.Pcw[2];
    double pcu, pcv;
    world2cam(a.cam, pf0, pf1, pf2, pcu, pcv);
    const Bilinear bw = bilinear_setup(pcu, pcv, level);
    const float2 Pv = *reinterpret_cast<const float2 *>(a.warp_patch + (size_t)i * 64 * a.levels + 64 * level + 2 * lane);
    const long sw = (long)scale * width;
    double sq = 0.0;
#pragma unroll
    for (int k = 0; k < 2; k++) {
      const int pix = 2 * lane + k, x = pix >> 3, y = pix & 7;
      const long b = (long)(bw.v_ref_i + x * scale - 4 * scale) * width + (bw.u_ref_i - 4 * scale) + (long)y * scale;
      const float cur = bil(bw.w_tl, bw.w_tr, bw.w_bl, bw.w_br, tap(a.img, b, npix), tap(a.img, b + scale, npix), tap(a.img, b + sw, npix), tap(a.img, b + sw + scale, npix));
      const double res = (double)__fsub_rn(cur, k == 0 ? Pv.x : Pv.y);  // float residual, then widened (:1466-1468)
      const double *hi6 = v.H_sub_inv + ((size_t)lp * 64 + pix) * 6;
      const double r0 = hi6[0], r1 = hi6[1], r2 = hi6[2], t0 = hi6[3], t1 = hi6[4], t2 = hi6[5];
      // q = J_dt * [Pwi]x ; JdR = J_dR * Rwi + q * Rwi ; Jdt = J_dt * Rwi   (:1471-1472, same association)
      const double q0 = t1 * Pwi[2] - t2 * Pwi[1], q1 = -t0 * Pwi[2] + t2 * Pwi[0], q2 = t0 * Pwi[1] - t1 * Pwi[0];
      double row[8];
#pragma unroll
      for (int c = 0; c < 3; c++) {
        row[c] = (r0 * Rwi[c] + r1 * Rwi[3 + c] + r2 * Rwi[6 + c]) + (q0 * Rwi[c] + q1 * Rwi[3 + c] + q2 * Rwi[6 + c]);
        row[3 + c] = t0 * Rwi[c] + t1 * Rwi[3 + c] + t2 * Rwi[6 + c];
      }
      row[6] = 0.0, row[7] = res;
      double4 *dst = reinterpret_cast<double4 *>(&sm.rows[warp][pix][0]);
      dst[0] = make_double4(row[0], row[1], row[2], row[3]);
      dst[1] = make_double4(row[4], row[5], row[6], row[7]);
      sq += res * res;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if (lane == 0) a.errors[i] = (float)sq;
    n_meas += 64.0;
    __syncwarp();
    {
      const int g = lane >> 2, t = lane & 3;
#pragma unroll
      for (int s = 0; s < 16; s++) {
        const double val = sm.rows[warp][4 * s + t][g];
        dmma_m8n8k4(D0, D1, val, val);
      }
    }
    __syncwarp();
  }
}

// One iteration of updateStateInverse's measurement build at pyramid level a.level.
__global__ void __launch_bounds__(VIO_THREADS, 1) vio_inverse_patch_kernel(const VioKernelArgs a, const VioInvArgs v) {
  if (a.slot_iter > 0 && a.ctrl->level_done) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  VioSmem &sm = *reinterpret_cast<VioSmem *>(smem_raw);
  vio_pose_consts(sm, a, a.state);
  double D0 = 0.0, D1 = 0.0, n_meas = 0.0;
  int lo, hi;
  vio_block_range(a.count, lo, hi);
  vio_inverse_process_range(a, v, sm, a.level, lo, hi, a.state, D0, D1, n_meas);
  reduce_info<VIO_WARPS, 7>(sm.red, D0, D1, n_meas, a.partials, a.partial_stride, a.info, a.ctrl);
}

}  // namespace esikf
