// Host side of the C ABI declared in include/esikf_b200.h: context, device mirror of the voxel map, staging of the
// per-tick inputs, and the launch sequences of the LIO / VIO update loops. No CPU fallback: every entry point fails
// with a status code when the device or an input is missing.
#include <cuda.h>
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <utility>
#include <vector>

#include "esikf_dev.cuh"

// single translation unit: the kernels are included so the whole library builds with one nvcc invocation
#include "esikf_lio.cu"
#include "esikf_solve.cu"
#include "esikf_vio.cu"
#include "esikf_fused.cu"
#include "esikf_map.cu"

using namespace esikf;

// ---------------------------------------------------------------------------------------------------------------------
// NCCL through dlopen: the library has no link-time dependency on NCCL; when the process already holds a libnccl.so.2
// (e.g. torch's bundled one) that copy is reused.
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
  void *handle = nullptr;
  int (*GetUniqueId)(ncclUniqueId *) = nullptr;
  int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  bool load() {
    if (handle) return true;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
      handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD);
      if (handle) break;
    }
    if (!handle)
      for (const char *n : names) {
        handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (handle) break;
      }
    if (!handle) return false;
    GetUniqueId = (int (*)(ncclUniqueId *))dlsym(handle, "ncclGetUniqueId");
    CommInitRank = (int (*)(ncclComm_t *, int, ncclUniqueId, int))dlsym(handle, "ncclCommInitRank");
    AllReduce = (int (*)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(handle, "ncclAllReduce");
    CommDestroy = (int (*)(ncclComm_t))dlsym(handle, "ncclCommDestroy");
    GetErrorString = (const char *(*)(int))dlsym(handle, "ncclGetErrorString");
    return GetUniqueId && CommInitRank && AllReduce && CommDestroy;
  }
};
static NcclApi g_nccl;
enum { NCCL_FLOAT64 = 8, NCCL_SUM = 0 };

// ---------------------------------------------------------------------------------------------------------------------
// Device array that owns its memory: grows (contents discarded) on reserve, freed with its owner.
template <typename T> struct DevBuf {
  T *p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr, o.cap = 0; }
  DevBuf &operator=(DevBuf &&o) noexcept {
    std::swap(p, o.p), std::swap(cap, o.cap);
    return *this;
  }
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr, cap = 0;
    size_t want = n + n / 4 + 64;
    cudaError_t e = cudaMalloc(&p, want * sizeof(T));
    if (e == cudaSuccess) cap = want;
    return e;
  }
  // reserve `reserve_n` elements, then copy the first `n` from the host on `st` (nothing when n == 0)
  cudaError_t upload(const T *src, size_t n, size_t reserve_n, cudaStream_t st) {
    cudaError_t e = reserve(reserve_n);
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(p, src, n * sizeof(T), cudaMemcpyHostToDevice, st);
    return e;
  }
};

// One arena of the device-resident voxel map. The context holds two: esikf_map_device_slide copies the surviving roots
// into the spare one, then the two change roles. A host-uploaded map (esikf_map_upload) uses slots, planes and recs only.
struct MapStorage {
  DevBuf<HashSlot> slots;
  DevBuf<int> slot_root, slot_cap;
  DevBuf<MapNode> nodes;
  DevBuf<double> pool;
  DevBuf<PlaneRec> recs;        // what the residual kernel reads (144-byte records derived on the device)
  DevBuf<esikf_plane> planes;   // the map as uploaded / refitted (256-byte records)
  DevBuf<int> rec_node, counters;
  DevBuf<unsigned long long> counters64;
  uint32_t hash_cap = 0;
  int node_cap = 0, rec_cap = 0;
  long long pool_cap = 0;
  cudaError_t reserve(uint32_t hashes, int nodes_n, int recs_n, long long points) {
    cudaError_t e;
    if ((e = slots.reserve(hashes)) || (e = slot_root.reserve(hashes)) || (e = slot_cap.reserve(hashes)) || (e = nodes.reserve((size_t)nodes_n)) ||
        (e = pool.reserve((size_t)points * MAP_PT_D)) || (e = recs.reserve((size_t)recs_n)) || (e = planes.reserve((size_t)recs_n)) ||
        (e = rec_node.reserve((size_t)recs_n)) || (e = counters.reserve(8)) || (e = counters64.reserve(2)))
      return e;
    hash_cap = hashes, node_cap = nodes_n, rec_cap = recs_n, pool_cap = points;
    return cudaSuccess;
  }
  MapArena arena(const MapCfg &cfg) const {
    MapArena A{};
    A.slots = slots.p, A.hash_mask = hash_cap - 1, A.slot_root = slot_root.p, A.slot_cap = slot_cap.p;
    A.nodes = nodes.p, A.node_cap = node_cap, A.pool = pool.p, A.pool_cap = pool_cap;
    A.recs = recs.p, A.planes = planes.p, A.rec_node = rec_node.p, A.rec_cap = rec_cap;
    A.counters = counters.p, A.counters64 = counters64.p, A.cfg = cfg;
    return A;
  }
};

// Loop-control block shared by the kernels of one update. The persistent kernels initialise it from CTA 0; the
// per-iteration launch path zeroes it with a memset.
struct CtlBlock {
  esikf_lio_stats lio_stats;
  Ctrl ctrl;
  unsigned char pad[64];
  esikf_vio_stats vio_stats;
};
static_assert(offsetof(CtlBlock, ctrl) == sizeof(esikf_lio_stats) && offsetof(CtlBlock, vio_stats) == sizeof(esikf_lio_stats) + sizeof(Ctrl) + 64 &&
                  sizeof(CtlBlock) == sizeof(esikf_lio_stats) + sizeof(Ctrl) + 64 + sizeof(esikf_vio_stats),
              "control block layout [esikf_lio_stats | Ctrl | 64 B pad | esikf_vio_stats]");

#define VIO_PERSIST_SMEM (sizeof(VioSmem) + sizeof(FusedSolveSmem))

struct esikf_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  std::string err;
  int64_t launches = 0;
  int solve_mode = 0;
  int loop_mode = 2;      // >= 1: one persistent cooperative kernel per update (gain solve replicated in every CTA, one grid
                          //    barrier per iteration; carries the NVLink peer exchange when peers are attached),
                          // 0: one residual + one solve launch per iteration (NCCL communicator, kernel timing)
  int coop_ok = 0;
  int coop_lio = 0, coop_vio = 0;  // co-resident CTAs per SM of the persistent kernels
  uint32_t tuning = 0;             // ESIKF_TUNE_* flags (measurement variants)
  DevBuf<unsigned int> barrier;       // two grid barriers {counter @ +0, release word @ +128 B}, 256 B apart; launches alternate
  DevBuf<unsigned long long> stamps;  // 8 per slot: 8 LIO slots then 64 VIO slots
  bool want_stamps = false;
  esikf_extrinsics ext{};
  bool have_ext = false, have_ext_dev = false;
  double ext_host[12] = {};

  // map
  MapStorage map, map_spare;
  uint32_t hash_mask = 0;
  DevBuf<int32_t> patch_ids;
  int n_planes = 0, n_roots = 0;
  double voxel_size = 0.5;
  bool have_map = false;

  // device-resident map (esikf_map_device_*): octree nodes, point lists and refits stay on the GPU
  bool dev_map = false;
  esikf_map_cfg map_cfg{};
  MapCfg map_kcfg{};           // map_cfg as the map kernels read it
  DevBuf<int> map_work, map_survivors;
  DevBuf<double> map_pt, map_pt_normal;
  DevBuf<unsigned int> map_key_in, map_key_out, map_idx_in, map_idx_out;
  DevBuf<MapTouched> map_touched;
  DevBuf<unsigned char> map_sort_tmp;
  int map_pt_n = 0;            // points the normal snapshot / last map step covers
  bool map_normals_valid = false;
  int map_hash_bits = 0;
  esikf_map_stats map_last{};

  // LIO
  DevBuf<float> pts;
  DevBuf<double> pre;
  DevBuf<int32_t> match_plane, normal_plane;
  DevBuf<float> dis;
  int n_pts = 0;
  int pre_stride = 0;
  bool scan_fresh = false;   // precompute pending
  esikf_lio_cfg lio_cfg{};
  DevBuf<double> ext_dev;    // extR(9) extT(3)

  // shared update state
  DevBuf<double> state_prop;             // [state 386 | prop 386] contiguous: one H2D copy per update
  double *state = nullptr, *prop = nullptr;
  DevBuf<double> info, partials, old_state, G;
  // pinned staging ring for the two packed states of an update (slot reuse guarded by an event)
  enum { STAGE_SLOTS = 16 };
  double *stage = nullptr;
  unsigned char *stage_ctrl = nullptr;   // pinned copy of the loop-control block read by the fetch calls
  cudaEvent_t stage_ev[STAGE_SLOTS] = {};
  unsigned stage_idx = 0;
  unsigned launch_parity = 0;            // the persistent kernels alternate between two grid-barrier counters
  DevBuf<CtlBlock> ctl;
  int partial_blocks = 0;

  // VIO
  esikf_camera cam{};
  esikf_vio_cfg vio_cfg{};
  bool have_cam = false;
  DevBuf<uint8_t> img;
  int img_w = 0, img_h = 0;
  VioTma tma;                      // tensor maps of `img` (ESIKF_TUNE_VIO_TMA), encoded for tma_img / tma_w x tma_h
  const uint8_t *tma_img = nullptr;
  int tma_w = 0, tma_h = 0;
  DevBuf<double> vis_pos, inv_expo;
  DevBuf<float> warp_patch, errors;
  DevBuf<int32_t> search_levels;
  DevBuf<double> inv_ref_px, inv_ref_f, inv_ref_R, inv_ref_pos, H_sub_inv;  // inverse-compositional variant
  DevBuf<int32_t> inv_ref_idx;
  int n_inv_refs = 0;
  DevBuf<float> warp_out;        // esikf_vio_warp_affine scratch (does not disturb the installed patches)
  DevBuf<int32_t> warp_levels;
  int n_patches = 0;
  // warp producers
  std::vector<DevBuf<uint8_t>> ref_imgs;
  DevBuf<const uint8_t *> ref_img_ptrs;
  int ref_w = 0, ref_h = 0;
  DevBuf<int32_t> ref_idx;
  DevBuf<double> px_ref, pos_w, normal_w, T_ref, T_cur, A_cur_ref, pc_buf;
  DevBuf<float> patch_buf;

  // multi-GPU
  int rank = 0, nranks = 1;
  ncclComm_t comm = nullptr;
  // NVLink peer-memory all-reduce inside the persistent kernels
  unsigned long long *mailbox = nullptr;             // own mailbox [2][PEER_MAX_RANKS][PEER_SLOT_WORDS], followed by the exchange counter
  std::vector<unsigned long long *> peer_ptrs;       // mailbox of every rank as mapped into this process
  DevBuf<unsigned long long *> peer_ptrs_dev;
  bool p2p = false;
  unsigned int *peer_seq_dev = nullptr;              // device word: peer exchanges executed so far

  // measurement
  bool timing = false;
  std::vector<cudaEvent_t> ev;      // 3 per slot: before residual, after residual, after solve
  int lio_slots = 0, vio_slots = 0;
  bool lio_timed = false, vio_timed = false;
  cudaEvent_t prof_ev[2] = {};      // esikf_profile_kernel
  DevBuf<uint8_t> flush;
  DevBuf<double> scratch_state, point_cov_tmp;

  // the device buffers free themselves; this releases what is not a DevBuf (the caller has made `device` current)
  ~esikf_ctx() {
    if (stream) cudaStreamSynchronize(stream);
    if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
    for (size_t r = 0; r < peer_ptrs.size(); r++)
      if ((int)r != rank && peer_ptrs[r]) cudaIpcCloseMemHandle(peer_ptrs[r]);
    if (mailbox) cudaFree(mailbox);
    if (stage) cudaFreeHost(stage);
    if (stage_ctrl) cudaFreeHost(stage_ctrl);
    for (cudaEvent_t e : stage_ev)
      if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : prof_ev)
      if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
    if (stream) cudaStreamDestroy(stream);
  }
};

static int fail(esikf_ctx *c, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}
#define CK(call)                                                                                                   \
  do {                                                                                                             \
    cudaError_t e__ = (call);                                                                                      \
    if (e__ != cudaSuccess) return fail(ctx, ESIKF_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

static cudaEvent_t *timing_events(esikf_ctx *ctx, int base, int slot) {
  size_t need = (size_t)(base + slot + 1) * 3;
  while (ctx->ev.size() < need) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    ctx->ev.push_back(e);
  }
  return &ctx->ev[(size_t)(base + slot) * 3];
}
enum { EV_LIO_BASE = 0, EV_VIO_BASE = 8 };

static void shard_of(int n, int rank, int nranks, int &begin, int &count) {
  // contiguous blocks, remainder spread over the first ranks
  int base = n / nranks, rem = n % nranks;
  begin = rank * base + (rank < rem ? rank : rem);
  count = base + (rank < rem ? 1 : 0);
}

extern "C" {

int esikf_create(esikf_ctx **out, int device) {
  if (!out) return ESIKF_ERR_ARG;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return ESIKF_ERR_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return ESIKF_ERR_NO_DEVICE;
  if (prop.major != 10) return ESIKF_ERR_NO_DEVICE;  // sm_100a binary only
  esikf_ctx *ctx = new esikf_ctx;
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return ESIKF_ERR_CUDA;
  }
  bool ok = ctx->state_prop.reserve(2 * S_N) == cudaSuccess && ctx->info.reserve(NE_MAX) == cudaSuccess &&
            cudaMallocHost(&ctx->stage, (size_t)esikf_ctx::STAGE_SLOTS * 2 * S_N * sizeof(double)) == cudaSuccess &&
            cudaMallocHost(&ctx->stage_ctrl, 256) == cudaSuccess &&
            ctx->old_state.reserve(32) == cudaSuccess && ctx->G.reserve(19 * 7) == cudaSuccess &&
            ctx->ctl.reserve(1) == cudaSuccess && ctx->ext_dev.reserve(12) == cudaSuccess && ctx->scratch_state.reserve(S_N) == cudaSuccess;
  ctx->partial_blocks = ctx->sm_count < 160 ? ctx->sm_count : 160;  // persistent residual kernels: one CTA per SM
  ok = ok && ctx->partials.reserve((size_t)2 * ctx->partial_blocks * NE_MAX) == cudaSuccess && ctx->stamps.reserve(8 * 72 + 64 + 160) == cudaSuccess &&
       ctx->barrier.reserve(128) == cudaSuccess;
  if (ok) cudaMemsetAsync(ctx->barrier.p, 0, 128 * sizeof(unsigned int), ctx->stream);
  if (ok) {
    ctx->state = ctx->state_prop.p, ctx->prop = ctx->state_prop.p + S_N;
    for (int i = 0; i < esikf_ctx::STAGE_SLOTS; i++) ok = ok && cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming) == cudaSuccess;
    for (cudaEvent_t &e : ctx->prof_ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
  }
  if (ok) cudaMemsetAsync(ctx->ctl.p, 0, sizeof(CtlBlock), ctx->stream);
  cudaDeviceGetAttribute(&ctx->coop_ok, cudaDevAttrCooperativeLaunch, device);
  if (!ok) {
    delete ctx;
    return ESIKF_ERR_CUDA;
  }
  cudaFuncSetAttribute(lio_residual_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(LioSmem));
  cudaFuncSetAttribute(vio_patch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(VioSmem));
  cudaFuncSetAttribute(vio_inverse_patch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(VioSmem));
  cudaError_t ea = cudaFuncSetAttribute(lio_update_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(LioSmem));
  cudaFuncSetAttribute(lio_update_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(LioSmem));
  cudaError_t eb = cudaFuncSetAttribute(vio_update_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VIO_PERSIST_SMEM);
  cudaFuncSetAttribute(vio_update_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VIO_PERSIST_SMEM);
  cudaFuncSetAttribute(vio_update_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VIO_PERSIST_SMEM);
  cudaFuncSetAttribute(vio_update_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VIO_PERSIST_SMEM);
  // the persistent kernels need every CTA co-resident: check what the device can hold
  int occ_l = 0, occ_v = 0, occ_lp = 0, occ_vp = 0, occ_r = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_l, lio_update_kernel<false>, LIO_THREADS, sizeof(LioSmem));
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_lp, lio_update_kernel<true>, LIO_THREADS, sizeof(LioSmem));
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_v, vio_update_kernel<false, false>, VIO_THREADS, VIO_PERSIST_SMEM);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_vp, vio_update_kernel<true, true>, VIO_THREADS, VIO_PERSIST_SMEM);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_r, lio_residual_kernel, LIO_THREADS, sizeof(LioSmem));
  ctx->coop_lio = occ_l < occ_lp ? occ_l : occ_lp, ctx->coop_vio = occ_v < occ_vp ? occ_v : occ_vp;
  if (getenv("ESIKF_DEBUG")) {
    fprintf(stderr, "[esikf] SMs=%d smem LIO=%zu VIO=%zu attr=%d/%d occupancy: lio_update=%d vio_update=%d lio_residual=%d coop=%d\n", ctx->sm_count, sizeof(LioSmem),
            VIO_PERSIST_SMEM, (int)ea, (int)eb, occ_l, occ_v, occ_r, ctx->coop_ok);
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, lio_residual_kernel);
    fprintf(stderr, "[esikf] lio_residual: regs=%d local=%zu\n", fa.numRegs, fa.localSizeBytes);
    cudaFuncGetAttributes(&fa, lio_update_kernel<false>);
    fprintf(stderr, "[esikf] lio_update: regs=%d local=%zu\n", fa.numRegs, fa.localSizeBytes);
    cudaFuncGetAttributes(&fa, vio_update_kernel<false, false>);
    fprintf(stderr, "[esikf] vio_update: regs=%d local=%zu\n", fa.numRegs, fa.localSizeBytes);
  }
  cudaGetLastError();
  *out = ctx;
  return ESIKF_OK;
}

void esikf_destroy(esikf_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  delete ctx;
}

const char *esikf_last_error(const esikf_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
void *esikf_stream(esikf_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
int64_t esikf_launch_count(const esikf_ctx *ctx) { return ctx ? ctx->launches : 0; }

void *esikf_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (bytes == 0 || cudaMallocHost(&p, bytes) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void esikf_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

int esikf_synchronize(esikf_ctx *ctx) {
  if (!ctx) return ESIKF_ERR_ARG;
  CK(cudaStreamSynchronize(ctx->stream));
  return ESIKF_OK;
}
int esikf_set_solve_mode(esikf_ctx *ctx, int mode) {
  if (!ctx || mode < 0 || mode > 1) return ESIKF_ERR_ARG;
  ctx->solve_mode = mode;
  return ESIKF_OK;
}
int esikf_set_loop_mode(esikf_ctx *ctx, int mode) {
  if (!ctx || mode < 0 || mode > 2) return ESIKF_ERR_ARG;  // 1 and 2 both select the persistent kernels
  ctx->loop_mode = mode;
  return ESIKF_OK;
}
int esikf_set_tuning(esikf_ctx *ctx, uint32_t flags) {
  if (!ctx || (flags & ~(uint32_t)(ESIKF_TUNE_STAGE_LDG | ESIKF_TUNE_VIO_TMA))) return ESIKF_ERR_ARG;
  ctx->tuning = flags;
  return ESIKF_OK;
}
int esikf_set_extrinsics(esikf_ctx *ctx, const esikf_extrinsics *ext) {
  if (!ctx || !ext) return ESIKF_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->ext = *ext;
  ctx->have_ext = true;
  double h[12];
  memcpy(h, ext->extR, 9 * sizeof(double));
  memcpy(h + 9, ext->extT, 3 * sizeof(double));
  if (ctx->have_ext_dev && memcmp(h, ctx->ext_host, sizeof(h)) == 0) return ESIKF_OK;  // unchanged (the shim sets it every tick): nothing to do
  CK(cudaMemcpyAsync(ctx->ext_dev.p, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));  // `h` is a stack buffer
  memcpy(ctx->ext_host, h, sizeof(h));
  ctx->have_ext_dev = true;
  return ESIKF_OK;
}

int esikf_set_lidar_extrinsics(esikf_ctx *ctx, const double extR[9], const double extT[3]) {
  if (!ctx || !extR || !extT) return ESIKF_ERR_ARG;
  esikf_extrinsics e = ctx->ext;
  if (!ctx->have_ext) {
    memset(&e, 0, sizeof(e));
    e.Rcl[0] = e.Rcl[4] = e.Rcl[8] = 1.0;
  }
  memcpy(e.extR, extR, sizeof(e.extR));
  memcpy(e.extT, extT, sizeof(e.extT));
  return esikf_set_extrinsics(ctx, &e);
}

// ---------------------------------------------------------------------------------------------------------------- map
int esikf_map_upload(esikf_ctx *ctx, const int64_t *keys, const int32_t *first, const int32_t *count, int32_t n_roots,
                     const esikf_plane *planes, int32_t n_planes, double voxel_size) {
  if (!ctx || n_roots < 0 || n_planes < 0 || (n_roots > 0 && (!keys || !first || !count)) || (n_planes > 0 && !planes) || !(voxel_size > 0))
    return fail(ctx, ESIKF_ERR_ARG, "map_upload: bad argument");
  CK(cudaSetDevice(ctx->device));
  uint32_t cap = 1024;
  while (cap < (uint32_t)n_roots * 2u) cap <<= 1;
  std::vector<HashSlot> table(cap);
  for (auto &s : table) s.key = ESIKF_KEY_EMPTY, s.first = 0, s.count = 0;
  for (int r = 0; r < n_roots; r++) {
    long long x = keys[3 * r], y = keys[3 * r + 1], z = keys[3 * r + 2];
    if (!key_in_range(x, y, z)) return fail(ctx, ESIKF_ERR_ARG, "map_upload: voxel key (%lld,%lld,%lld) outside +-2^20", x, y, z);
    if (first[r] < 0 || count[r] < 0 || first[r] + count[r] > n_planes) return fail(ctx, ESIKF_ERR_ARG, "map_upload: root %d plane range", r);
    unsigned long long k = pack_key(x, y, z);
    uint32_t s = hash_key(k) & (cap - 1);
    while (table[s].key != ESIKF_KEY_EMPTY) {
      if (table[s].key == k) return fail(ctx, ESIKF_ERR_ARG, "map_upload: duplicate voxel key");
      s = (s + 1) & (cap - 1);
    }
    table[s].key = k, table[s].first = (uint32_t)first[r], table[s].count = (uint32_t)count[r];
  }
  MapStorage &M = ctx->map;
  CK(M.slots.reserve(cap));
  CK(M.planes.reserve((size_t)n_planes + 1));
  CK(M.recs.reserve((size_t)n_planes + 1));
  CK(cudaMemcpyAsync(M.slots.p, table.data(), cap * sizeof(HashSlot), cudaMemcpyHostToDevice, ctx->stream));
  if (n_planes) {
    CK(cudaMemcpyAsync(M.planes.p, planes, (size_t)n_planes * sizeof(esikf_plane), cudaMemcpyHostToDevice, ctx->stream));
    plane_compact_kernel<<<(n_planes + 127) / 128, 128, 0, ctx->stream>>>(M.planes.p, nullptr, n_planes, M.recs.p);
    ctx->launches++;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->hash_mask = cap - 1;
  ctx->n_planes = n_planes, ctx->n_roots = n_roots;
  ctx->voxel_size = voxel_size;
  ctx->have_map = true;
  ctx->dev_map = false;  // a host-flattened map replaces a device-resident one
  return ESIKF_OK;
}

int esikf_map_patch(esikf_ctx *ctx, const int32_t *plane_ids, const esikf_plane *planes, int32_t n) {
  if (!ctx || n < 0 || (n > 0 && (!plane_ids || !planes))) return fail(ctx, ESIKF_ERR_ARG, "map_patch: bad argument");
  if (!ctx->have_map) return fail(ctx, ESIKF_ERR_STATE, "map_patch before map_upload");
  if (ctx->dev_map) return fail(ctx, ESIKF_ERR_STATE, "map_patch: the map is device-resident (esikf_map_device_init); it refits itself");
  CK(cudaSetDevice(ctx->device));
  for (int i = 0; i < n; i++)
    if (plane_ids[i] < 0 || plane_ids[i] >= ctx->n_planes) return fail(ctx, ESIKF_ERR_ARG, "map_patch: plane id %d", plane_ids[i]);
  for (int i = 0; i < n;) {
    int j = i + 1;
    while (j < n && plane_ids[j] == plane_ids[j - 1] + 1) j++;  // a run of consecutive ids travels as one copy
    CK(cudaMemcpyAsync(ctx->map.planes.p + plane_ids[i], planes + i, (size_t)(j - i) * sizeof(esikf_plane), cudaMemcpyHostToDevice, ctx->stream));
    i = j;
  }
  if (n > 0) {
    CK(ctx->patch_ids.upload(plane_ids, n, n, ctx->stream));
    plane_compact_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->map.planes.p, ctx->patch_ids.p, n, ctx->map.recs.p);
    ctx->launches++;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return ESIKF_OK;
}

// ------------------------------------------------------------------------------------------------ device-resident map (f1)
static int map_check_errors(esikf_ctx *ctx, const char *what) {
  int c[4];
  unsigned long long pool_used = 0;
  CK(cudaMemcpyAsync(c, ctx->map.counters.p, sizeof(c), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(&pool_used, ctx->map.counters64.p, sizeof(pool_used), cudaMemcpyDeviceToHost, ctx->stream));
  int work[2];
  CK(cudaMemcpyAsync(work, ctx->map_work.p, sizeof(work), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->map_last.nodes = c[0], ctx->map_last.records = c[1], ctx->map_last.errors = c[2], ctx->map_last.roots = c[3];
  ctx->map_last.pool_points = (int64_t)pool_used, ctx->map_last.touched_roots = work[0];
  ctx->n_planes = c[1] < ctx->map.rec_cap ? c[1] : ctx->map.rec_cap;
  ctx->n_roots = c[3];
  if (c[2]) {
    ctx->have_map = false;  // the map is not trustworthy any more: the next lio_run must not use it
    return fail(ctx, ESIKF_ERR_STATE, "%s: device map capacity exceeded (flags 0x%x:%s%s%s%s%s%s) — raise the esikf_map_cfg capacities and rebuild", what, c[2],
                (c[2] & MAP_ERR_NODES) ? " nodes" : "", (c[2] & MAP_ERR_POOL) ? " point-pool" : "", (c[2] & MAP_ERR_RECS) ? " records" : "",
                (c[2] & MAP_ERR_HASH) ? " hash" : "", (c[2] & MAP_ERR_KEY) ? " key-range" : "", (c[2] & MAP_ERR_STACK) ? " octree-depth" : "");
  }
  return ESIKF_OK;
}

int esikf_map_device_init(esikf_ctx *ctx, const esikf_map_cfg *cfg) {
  if (!ctx || !cfg || !(cfg->voxel_size > 0) || cfg->max_layer < 0 || cfg->max_layer >= MAP_MAX_LAYERS || cfg->max_points_num < 1)
    return fail(ctx, ESIKF_ERR_ARG, "map_device_init: bad argument");
  for (int k = 0; k <= cfg->max_layer; k++)
    if (cfg->layer_init_num[k] < 1) return fail(ctx, ESIKF_ERR_ARG, "map_device_init: layer_init_num[%d] = %d", k, cfg->layer_init_num[k]);
  CK(cudaSetDevice(ctx->device));
  const int64_t roots = cfg->root_capacity > 0 ? cfg->root_capacity : (1 << 20);
  uint32_t cap = 1024;
  int bits = 10;
  while ((int64_t)cap < 2 * roots) cap <<= 1, bits++;
  const int64_t node_cap = cfg->node_capacity > 0 ? cfg->node_capacity : 4 * roots;
  const int64_t rec_cap = cfg->record_capacity > 0 ? cfg->record_capacity : 4 * roots;
  const int64_t pool_cap = cfg->point_capacity > 0 ? cfg->point_capacity : 64 * roots;
  if (node_cap > 0x7fffffff || rec_cap > 0x7fffffff || pool_cap > 0x7fffffff) return fail(ctx, ESIKF_ERR_ARG, "map_device_init: capacity above 2^31");
  CK(ctx->map.reserve(cap, (int)node_cap, (int)rec_cap, pool_cap));
  CK(ctx->map_work.reserve(4));
  MapCfg &K = ctx->map_kcfg;
  K.voxel_size = (float)cfg->voxel_size, K.planer_threshold = (float)cfg->min_eigen_value;
  K.max_layer = cfg->max_layer, K.max_points_num = cfg->max_points_num;
  for (int k = 0; k < MAP_MAX_LAYERS; k++) K.layer_init_num[k] = cfg->layer_init_num[k <= cfg->max_layer ? k : cfg->max_layer];
  map_reset_kernel<<<(cap + 255) / 256, 256, 0, ctx->stream>>>(ctx->map.arena(K));
  CK(cudaMemsetAsync(ctx->map_work.p, 0, 4 * sizeof(int), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->launches++;
  ctx->map_cfg = *cfg;
  ctx->map_hash_bits = bits;
  ctx->hash_mask = cap - 1;
  ctx->voxel_size = cfg->voxel_size;
  ctx->n_planes = 0, ctx->n_roots = 0;
  ctx->dev_map = true, ctx->have_map = true;  // an empty map is a valid map (nothing matches)
  ctx->map_normals_valid = false;
  memset(&ctx->map_last, 0, sizeof(ctx->map_last));
  return ESIKF_OK;
}

// sort by slot, list the touched roots, replay them
static int map_apply_points(esikf_ctx *ctx, int n, bool build) {
  cudaStream_t st = ctx->stream;
  const unsigned int invalid = ctx->map.hash_cap;
  size_t tmp_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, ctx->map_key_in.p, ctx->map_key_out.p, ctx->map_idx_in.p, ctx->map_idx_out.p, n, 0, ctx->map_hash_bits + 1, st);
  CK(ctx->map_sort_tmp.reserve(tmp_bytes + 16));
  CK(cub::DeviceRadixSort::SortPairs(ctx->map_sort_tmp.p, tmp_bytes, ctx->map_key_in.p, ctx->map_key_out.p, ctx->map_idx_in.p, ctx->map_idx_out.p, n, 0,
                                     ctx->map_hash_bits + 1, st));
  CK(cudaMemsetAsync(ctx->map_work.p, 0, 2 * sizeof(int), st));
  map_heads_kernel<<<(n + 255) / 256, 256, 0, st>>>(ctx->map_key_out.p, n, invalid, ctx->map_touched.p, ctx->map_work.p);
  map_replay_kernel<<<ctx->sm_count * 4, 128, 0, st>>>(ctx->map.arena(ctx->map_kcfg), ctx->map_touched.p, ctx->map_work.p, ctx->map_idx_out.p, ctx->map_pt.p, build ? 1 : 0);
  ctx->launches += 4;
  CK(cudaGetLastError());
  return map_check_errors(ctx, build ? "map_device_build" : "map_device_update");
}

static int map_reserve_tick(esikf_ctx *ctx, int n) {
  CK(ctx->map_pt.reserve((size_t)n * MAP_PT_D + 16));
  CK(ctx->map_pt_normal.reserve((size_t)n * 3 + 4));
  CK(ctx->map_key_in.reserve(n + 1));
  CK(ctx->map_key_out.reserve(n + 1));
  CK(ctx->map_idx_in.reserve(n + 1));
  CK(ctx->map_idx_out.reserve(n + 1));
  CK(ctx->map_touched.reserve(n + 1));
  return ESIKF_OK;
}

static int map_from_scan(esikf_ctx *ctx, const double *state, bool build) {
  if (!ctx) return ESIKF_ERR_ARG;
  if (!ctx->dev_map) return fail(ctx, ESIKF_ERR_STATE, "map_device_%s before esikf_map_device_init", build ? "build" : "update");
  if (!ctx->have_ext) return fail(ctx, ESIKF_ERR_STATE, "map_device_%s before set_extrinsics", build ? "build" : "update");
  if (!build && ctx->scan_fresh) return fail(ctx, ESIKF_ERR_STATE, "map_device_update: the resident scan has not been through esikf_lio_run yet");
  if (build && ctx->map_last.roots > 0) return fail(ctx, ESIKF_ERR_STATE, "map_device_build needs an empty map (esikf_map_device_init resets it)");
  CK(cudaSetDevice(ctx->device));
  const int n = ctx->n_pts;
  if (n == 0) return ESIKF_OK;
  int rc = map_reserve_tick(ctx, n);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  const double *dev_state = ctx->state;  // the posterior the last update left on the device
  if (state) {
    CK(ctx->scratch_state.upload(state, S_N, S_N, st));
    dev_state = ctx->scratch_state.p;
  }
  MapPointArgs a;
  memset(&a, 0, sizeof(a));
  a.pts = ctx->pts.p, a.pre = ctx->pre.p, a.pre_stride = ctx->pre_stride, a.n = n, a.state = dev_state;
  memcpy(a.extR, ctx->ext.extR, 72), memcpy(a.extT, ctx->ext.extT, 24);
  a.build = build ? 1 : 0, a.dept_err = (float)ctx->map_cfg.dept_err, a.beam_err = (float)ctx->map_cfg.beam_err;
  a.match_plane = build ? nullptr : ctx->normal_plane.p, a.recs = ctx->map.recs.p, a.pt_normal = ctx->map_pt_normal.p;
  a.pt = ctx->map_pt.p, a.pt_slot = ctx->map_key_in.p, a.pt_idx = ctx->map_idx_in.p, a.invalid_slot = ctx->map.hash_cap;
  map_points_kernel<<<(n + 255) / 256, 256, 0, st>>>(ctx->map.arena(ctx->map_kcfg), a);
  ctx->map_pt_n = n, ctx->map_normals_valid = !build;
  return map_apply_points(ctx, n, build);
}

int esikf_map_device_build(esikf_ctx *ctx, const double *state) {
  if (ctx && !state) return fail(ctx, ESIKF_ERR_ARG, "map_device_build: the pose the scan is mapped with is required");
  return map_from_scan(ctx, state, true);
}
int esikf_map_device_update(esikf_ctx *ctx, const double *state) { return map_from_scan(ctx, state, false); }

int esikf_map_device_update_points(esikf_ctx *ctx, const double *point_w, const double *var, int32_t n) {
  if (!ctx || n < 0 || (n > 0 && (!point_w || !var))) return fail(ctx, ESIKF_ERR_ARG, "map_device_update_points: bad argument");
  if (!ctx->dev_map) return fail(ctx, ESIKF_ERR_STATE, "map_device_update_points before esikf_map_device_init");
  if (n == 0) return ESIKF_OK;
  CK(cudaSetDevice(ctx->device));
  int rc = map_reserve_tick(ctx, n);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  // [n][12] = point_w | var: two strided copies
  CK(cudaMemcpy2DAsync(ctx->map_pt.p, MAP_PT_D * sizeof(double), point_w, 3 * sizeof(double), 3 * sizeof(double), n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpy2DAsync(ctx->map_pt.p + 3, MAP_PT_D * sizeof(double), var, 9 * sizeof(double), 9 * sizeof(double), n, cudaMemcpyHostToDevice, st));
  map_keys_kernel<<<(n + 255) / 256, 256, 0, st>>>(ctx->map.arena(ctx->map_kcfg), ctx->map_pt.p, n, ctx->map_key_in.p, ctx->map_idx_in.p, ctx->map.hash_cap);
  ctx->launches++;
  ctx->map_normals_valid = false;
  return map_apply_points(ctx, n, false);
}

// mapSliding / clearMemOutOfMap (src/voxel_map.cpp:924-971)
int esikf_map_device_slide(esikf_ctx *ctx, const int64_t key_min[3], const int64_t key_max[3]) {
  if (!ctx) return ESIKF_ERR_ARG;
  if (!ctx->dev_map) return fail(ctx, ESIKF_ERR_STATE, "map_device_slide before esikf_map_device_init");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const MapStorage &M = ctx->map;
  const unsigned cap = M.hash_cap;
  CK(ctx->map_spare.reserve(cap, M.node_cap, M.rec_cap, M.pool_cap));
  CK(ctx->map_survivors.reserve((size_t)(ctx->map_last.roots > 0 ? ctx->map_last.roots : 1) + 1));
  const MapArena S = M.arena(ctx->map_kcfg), D = ctx->map_spare.arena(ctx->map_kcfg);
  const long long big = 1ll << 40;
  const long long lo[3] = {key_min ? key_min[0] : -big, key_min ? key_min[1] : -big, key_min ? key_min[2] : -big};
  const long long hi[3] = {key_max ? key_max[0] : big, key_max ? key_max[1] : big, key_max ? key_max[2] : big};
  map_reset_kernel<<<(cap + 255) / 256, 256, 0, st>>>(D);
  CK(cudaMemsetAsync(ctx->map_work.p, 0, 2 * sizeof(int), st));
  map_survivors_kernel<<<(cap + 255) / 256, 256, 0, st>>>(S, lo[0], lo[1], lo[2], hi[0], hi[1], hi[2], ctx->map_survivors.p, ctx->map_work.p);
  map_copy_kernel<<<ctx->sm_count * 4, 128, 0, st>>>(S, D, ctx->map_survivors.p, ctx->map_work.p);
  ctx->launches += 3;
  CK(cudaGetLastError());
  // the fresh arena becomes the map (also when the copy reports an error: the status says so and the map is invalidated)
  std::swap(ctx->map, ctx->map_spare);
  ctx->map_normals_valid = false;  // record positions of the last update are gone
  return map_check_errors(ctx, "map_device_slide");
}

int esikf_map_device_stats(esikf_ctx *ctx, esikf_map_stats *out) {
  if (!ctx || !out) return fail(ctx, ESIKF_ERR_ARG, "map_device_stats: bad argument");
  if (!ctx->dev_map) return fail(ctx, ESIKF_ERR_STATE, "map_device_stats before esikf_map_device_init");
  *out = ctx->map_last;
  return ESIKF_OK;
}

int esikf_map_device_download(esikf_ctx *ctx, int64_t *keys, int32_t *first, int32_t *count, int32_t roots_cap, esikf_plane *planes, int32_t planes_cap, int32_t *n_roots,
                              int32_t *n_planes) {
  if (!ctx || !n_roots || !n_planes) return fail(ctx, ESIKF_ERR_ARG, "map_device_download: bad argument");
  if (!ctx->dev_map) return fail(ctx, ESIKF_ERR_STATE, "map_device_download before esikf_map_device_init");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const bool fill = keys && first && count && planes && roots_cap > 0;
  DevBuf<long long> d_keys;
  DevBuf<int32_t> d_first, d_count;
  DevBuf<esikf_plane> d_planes;
  DevBuf<int> d_out;
  CK(d_out.reserve(2));
  CK(cudaMemsetAsync(d_out.p, 0, 2 * sizeof(int), st));
  if (fill) {
    CK(d_keys.reserve((size_t)roots_cap * 3));
    CK(d_first.reserve(roots_cap));
    CK(d_count.reserve(roots_cap));
    CK(d_planes.reserve(planes_cap > 0 ? planes_cap : 1));
  }
  const unsigned cap = ctx->map.hash_cap;
  map_download_kernel<<<(cap + 255) / 256, 256, 0, st>>>(ctx->map.arena(ctx->map_kcfg), fill ? d_keys.p : nullptr, d_first.p, d_count.p, d_planes.p, fill ? roots_cap : 0, fill ? planes_cap : 0, d_out.p);
  ctx->launches++;
  int out[2];
  CK(cudaMemcpyAsync(out, d_out.p, sizeof(out), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  *n_roots = out[0], *n_planes = out[1];
  int rc = ESIKF_OK;
  if (fill) {
    if (out[0] > roots_cap || out[1] > planes_cap)
      rc = fail(ctx, ESIKF_ERR_ARG, "map_device_download: %d roots / %d planes do not fit the buffers (%d / %d)", out[0], out[1], roots_cap, planes_cap);
    else {
      CK(cudaMemcpy(keys, d_keys.p, (size_t)out[0] * 3 * sizeof(int64_t), cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(first, d_first.p, (size_t)out[0] * sizeof(int32_t), cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(count, d_count.p, (size_t)out[0] * sizeof(int32_t), cudaMemcpyDeviceToHost));
      if (out[1]) CK(cudaMemcpy(planes, d_planes.p, (size_t)out[1] * sizeof(esikf_plane), cudaMemcpyDeviceToHost));
    }
  }
  return rc;
}

// pv.normal of every point of the last update (voxel_map.cpp:744: the plane that last became the point's best candidate in any
// iteration — normal_plane, not the final match; zero when there never was one): snapshotted by esikf_map_device_update
// before the records may move, otherwise gathered from the records now
__global__ void gather_normals_kernel(const int32_t *__restrict__ match_plane, const PlaneRec *__restrict__ recs, int n, double *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int m = match_plane[i];
  for (int k = 0; k < 3; k++) out[3 * (size_t)i + k] = m >= 0 ? recs[m].n[k] : 0.0;
}
int esikf_lio_fetch_normals(esikf_ctx *ctx, double *normals) {
  if (!ctx || !normals) return fail(ctx, ESIKF_ERR_ARG, "lio_fetch_normals: bad argument");
  if (!ctx->have_map || ctx->scan_fresh) return fail(ctx, ESIKF_ERR_STATE, "lio_fetch_normals before lio_run");
  CK(cudaSetDevice(ctx->device));
  const int n = ctx->n_pts;
  if (n == 0) return ESIKF_OK;
  if (!(ctx->dev_map && ctx->map_normals_valid && ctx->map_pt_n == n)) {
    CK(ctx->map_pt_normal.reserve((size_t)n * 3 + 4));
    gather_normals_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->normal_plane.p, ctx->map.recs.p, n, ctx->map_pt_normal.p);
    ctx->launches++;
  }
  CK(cudaMemcpyAsync(normals, ctx->map_pt_normal.p, (size_t)n * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return ESIKF_OK;
}

// ---------------------------------------------------------------------------------------------------------------- LIO
int esikf_lio_set_scan(esikf_ctx *ctx, const float *pts_xyz, int32_t n) {
  if (!ctx || n < 0 || (n > 0 && !pts_xyz)) return fail(ctx, ESIKF_ERR_ARG, "lio_set_scan: bad argument");
  CK(cudaSetDevice(ctx->device));
  ctx->pre_stride = (n + 31) & ~31;
  CK(ctx->pre.reserve((size_t)ctx->pre_stride * 9 + 16));
  CK(ctx->match_plane.reserve(n + 1));
  CK(ctx->normal_plane.reserve(n + 1));
  CK(ctx->dis.reserve(n + 1));
  CK(ctx->pts.upload(pts_xyz, (size_t)n * 3, (size_t)n * 3 + 4, ctx->stream));
  ctx->n_pts = n;
  ctx->scan_fresh = true;
  return ESIKF_OK;
}

static void lio_fill_args(esikf_ctx *ctx, LioKernelArgs &ka, double *state_ptr) {
  memset(&ka, 0, sizeof(ka));
  ka.pts = ctx->pts.p, ka.pre = ctx->pre.p;
  ka.pre_stride = ctx->pre_stride;
  ka.partial_stride = ctx->partial_blocks;
  shard_of(ctx->n_pts, ctx->rank, ctx->nranks, ka.begin, ka.count);
  ka.state = state_ptr, ka.prop = ctx->prop;
  ka.slots = ctx->map.slots.p, ka.hash_mask = ctx->hash_mask, ka.recs = ctx->map.recs.p;
  ka.stage_mode = (ctx->tuning & ESIKF_TUNE_STAGE_LDG) ? 1 : 0;
  memcpy(ka.extR, ctx->ext.extR, sizeof(ka.extR));
  memcpy(ka.extT, ctx->ext.extT, sizeof(ka.extT));
  ka.voxel_size = ctx->lio_cfg.voxel_size;
  ka.inv_voxel_size = 1.0 / ctx->lio_cfg.voxel_size;
  {
    int ex = 0;
    ka.inv_voxel_exact = (frexp(ctx->lio_cfg.voxel_size, &ex) == 0.5) ? 1 : 0;  // power of two: the reciprocal is exact
  }
  ka.voxel_size_f = (float)ctx->lio_cfg.voxel_size;
  ka.sigma_num = ctx->lio_cfg.sigma_num;
  ka.match_plane = ctx->match_plane.p, ka.normal_plane = ctx->normal_plane.p, ka.dis_to_plane = ctx->dis.p;
  ka.partials = ctx->partials.p, ka.info = ctx->info.p, ka.ctrl = &ctx->ctl.p->ctrl;
}
// the SolveArgs fields every solve launch sets; the LIO / VIO specific ones are the caller's
static SolveArgs solve_args(esikf_ctx *ctx, double *state_ptr, int max_iterations) {
  SolveArgs sa;
  memset(&sa, 0, sizeof(sa));
  sa.state = state_ptr, sa.prop = ctx->prop, sa.info = ctx->info.p, sa.ctrl = &ctx->ctl.p->ctrl;
  sa.max_iterations = max_iterations, sa.solve_mode = ctx->solve_mode;
  return sa;
}
static int lio_grid(const esikf_ctx *ctx, int count) {
  int chunks = (count + 31) / 32;  // whole warps are dealt to the CTAs: every SM takes part as soon as there is a warp for it
  int g = chunks < ctx->partial_blocks ? chunks : ctx->partial_blocks;
  return g < 1 ? 1 : g;
}
// Stage the two packed states of an update in pinned memory and upload them with ONE copy ([state | prop] is contiguous).
static int upload_states(esikf_ctx *ctx, const double *state_in, const double *state_prop) {
  const unsigned slot = ctx->stage_idx++ % esikf_ctx::STAGE_SLOTS;
  CK(cudaEventSynchronize(ctx->stage_ev[slot]));  // the copy that last used this slot has been consumed
  double *h = ctx->stage + (size_t)slot * 2 * S_N;
  memcpy(h, state_in, S_N * sizeof(double));
  memcpy(h + S_N, state_prop, S_N * sizeof(double));
  CK(cudaMemcpyAsync(ctx->state_prop.p, h, 2 * S_N * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaEventRecord(ctx->stage_ev[slot], ctx->stream));
  return ESIKF_OK;
}
// Whether an update runs as one persistent cooperative kernel (`coop`: co-resident CTAs per SM of that kernel).
static bool persistent_ok(const esikf_ctx *ctx, int coop) {
  return ctx->loop_mode >= 1 && (ctx->nranks == 1 || ctx->p2p) && ctx->coop_ok && coop > 0 && !ctx->timing;
}
// One cooperative launch of a persistent update kernel. `fn_solo` / `fn_peers` are its instantiations without and with
// the NVLink peer exchange; their parameters are (ka, sa, barrier, barrier_next, stamps, parity_stride, peer[, inv, tma]).
// The kernel's phase stamps go to `stamp_words` words at `stamps + stamp_off`.
static int launch_persistent(esikf_ctx *ctx, const char *name, const void *fn_solo, const void *fn_peers, int grid, int threads, size_t smem,
                             size_t stamp_off, size_t stamp_words, void *ka, SolveArgs *sa, void *inv, void *tma, bool &timed) {
  const unsigned par = ctx->launch_parity & 1;
  unsigned int *bar = ctx->barrier.p + 64 * par, *bar_next = ctx->barrier.p + 64 * (par ^ 1);  // this launch's barrier / the next launch's (zeroed by the kernel)
  unsigned long long *stamps = ctx->want_stamps ? ctx->stamps.p + stamp_off : nullptr;
  if (stamps) CK(cudaMemsetAsync(stamps, 0, stamp_words * sizeof(unsigned long long), ctx->stream));
  size_t parity_stride = (size_t)ctx->partial_blocks * NE_MAX;
  PeerArgs peer;
  peer.mbox = ctx->p2p ? ctx->peer_ptrs_dev.p : nullptr;
  peer.seq = ctx->peer_seq_dev;
  peer.rank = ctx->rank, peer.nranks = ctx->p2p ? ctx->nranks : 1;
  void *kargs[] = {ka, (void *)sa, (void *)&bar, (void *)&bar_next, (void *)&stamps, (void *)&parity_stride, (void *)&peer, inv, tma};
  const void *fn = (ctx->p2p && ctx->nranks > 1) ? fn_peers : fn_solo;
  cudaError_t le = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(threads), kargs, smem, ctx->stream);
  if (le != cudaSuccess) return fail(ctx, ESIKF_ERR_CUDA, "cooperative launch of %s failed: %s", name, cudaGetErrorString(le));
  ctx->launch_parity++;  // only a launch that happened consumes its barrier counter (the kernel zeroes the other one)
  ctx->launches += 1;
  timed = false;
  return ESIKF_OK;
}
static int allreduce_info(esikf_ctx *ctx) {
  if (ctx->nranks <= 1) return ESIKF_OK;
  if (!ctx->comm) return fail(ctx, ESIKF_ERR_STATE, "per-iteration launches with %d ranks need esikf_comm_init (NCCL)", ctx->nranks);
  int r = g_nccl.AllReduce(ctx->info.p, ctx->info.p, NE_MAX, NCCL_FLOAT64, NCCL_SUM, ctx->comm, ctx->stream);
  if (r != 0) return fail(ctx, ESIKF_ERR_COMM, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  return ESIKF_OK;
}

int esikf_lio_run(esikf_ctx *ctx, const double *state_in, const double *state_prop, const esikf_lio_cfg *cfg) {
  if (!ctx || !state_in || !state_prop || !cfg) return fail(ctx, ESIKF_ERR_ARG, "lio_run: null argument");
  if (!ctx->have_map) return fail(ctx, ESIKF_ERR_STATE, "lio_run before map_upload");
  if (!ctx->have_ext) return fail(ctx, ESIKF_ERR_STATE, "lio_run before set_extrinsics");
  ctx->map_normals_valid = false;  // a snapshot of pv.normal belongs to the update it was taken after
  if (cfg->max_iterations < 1 || cfg->max_iterations > 8) return fail(ctx, ESIKF_ERR_ARG, "lio_run: max_iterations must be in [1,8]");
  CK(cudaSetDevice(ctx->device));
  ctx->lio_cfg = *cfg;
  cudaStream_t st = ctx->stream;
  {
    int rc = upload_states(ctx, state_in, state_prop);
    if (rc) return rc;
  }
  const bool fused_lio = persistent_ok(ctx, ctx->coop_lio);
  // the persistent kernel initialises its own loop control / stats / barrier; the per-iteration path needs them zeroed
  if (!fused_lio) CK(cudaMemsetAsync(&ctx->ctl.p->lio_stats, 0, offsetof(CtlBlock, vio_stats), st));
  const int n = ctx->n_pts;
  if (ctx->scan_fresh) {
    if (n > 0) {
      lio_precompute_kernel<<<(n + 255) / 256, 256, 0, st>>>(ctx->pts.p, n, ctx->pre.p, ctx->pre_stride, ctx->ext_dev.p, (float)cfg->dept_err, (float)cfg->beam_err);
      ctx->launches++;
    }
    ctx->scan_fresh = false;
  }
  LioKernelArgs ka;
  lio_fill_args(ctx, ka, ctx->state);
  SolveArgs sa = solve_args(ctx, ctx->state, cfg->max_iterations);
  sa.lio_stats = &ctx->ctl.p->lio_stats;
  const int grid = lio_grid(ctx, ka.count);
  if (fused_lio)
    return launch_persistent(ctx, "lio_update_kernel", (const void *)lio_update_kernel<false>, (const void *)lio_update_kernel<true>, grid, LIO_THREADS,
                             sizeof(LioSmem), 0, 64, &ka, &sa, nullptr, nullptr, ctx->lio_timed);
  ctx->lio_timed = ctx->timing;
  ctx->lio_slots = cfg->max_iterations;
  for (int it = 0; it < cfg->max_iterations; it++) {
    cudaEvent_t *e = ctx->timing ? timing_events(ctx, EV_LIO_BASE, it) : nullptr;
    if (e) cudaEventRecord(e[0], st);
    ka.init_normal = (it == 0);
    lio_residual_kernel<<<grid, LIO_THREADS, sizeof(LioSmem), st>>>(ka);
    if (e) cudaEventRecord(e[1], st);
    int rc = allreduce_info(ctx);
    if (rc) return rc;
    lio_solve_kernel<<<1, SOLVE_THREADS, 0, st>>>(sa);
    if (e) cudaEventRecord(e[2], st);
    ctx->launches += 2;
  }
  CK(cudaGetLastError());
  return ESIKF_OK;
}

// Common tail of the fetch calls: bring the loop-control block along, synchronise, and turn an expired in-kernel wait
// (Ctrl::comm_error, sticky on the device) into ESIKF_ERR_COMM once.
static int finish_fetch(esikf_ctx *ctx) {
  Ctrl *h = reinterpret_cast<Ctrl *>(ctx->stage_ctrl);
  CK(cudaMemcpyAsync(h, &ctx->ctl.p->ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (h->comm_error) {
    cudaMemsetAsync(&ctx->ctl.p->ctrl.comm_error, 0, sizeof(int), ctx->stream);
    return fail(ctx, ESIKF_ERR_COMM, "a bounded in-kernel wait expired (grid barrier or peer mailbox): a rank did not take part in the update");
  }
  return ESIKF_OK;
}

int esikf_lio_fetch(esikf_ctx *ctx, double *state_out, esikf_lio_stats *stats, int32_t *match_plane, int32_t *normal_plane, float *dis_to_plane) {
  if (!ctx) return ESIKF_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t n = (size_t)ctx->n_pts;
  if (state_out) CK(cudaMemcpyAsync(state_out, ctx->state, S_N * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (stats) CK(cudaMemcpyAsync(stats, &ctx->ctl.p->lio_stats, sizeof(esikf_lio_stats), cudaMemcpyDeviceToHost, st));
  if (match_plane && n) CK(cudaMemcpyAsync(match_plane, ctx->match_plane.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (normal_plane && n) CK(cudaMemcpyAsync(normal_plane, ctx->normal_plane.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (dis_to_plane && n) CK(cudaMemcpyAsync(dis_to_plane, ctx->dis.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
  return finish_fetch(ctx);
}

int esikf_lio_update(esikf_ctx *ctx, const float *pts_xyz, int32_t n, const double *state_in, const double *state_prop, const esikf_lio_cfg *cfg,
                     double *state_out, esikf_lio_stats *stats, int32_t *match_plane, int32_t *normal_plane, float *dis_to_plane) {
  int rc = esikf_lio_set_scan(ctx, pts_xyz, n);
  if (rc) return rc;
  rc = esikf_lio_run(ctx, state_in, state_prop, cfg);
  if (rc) return rc;
  return esikf_lio_fetch(ctx, state_out, stats, match_plane, normal_plane, dis_to_plane);
}

__global__ void expand_point_cov_kernel(const double *__restrict__ pre, int pre_stride, int n, double *__restrict__ body_cov9, double *__restrict__ cross9) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double p[9];
  for (int k = 0; k < 9; k++) p[k] = pre[(size_t)k * pre_stride + i];
  if (body_cov9) {
    double *o = body_cov9 + 9 * (size_t)i;
    o[0] = p[3], o[1] = p[4], o[2] = p[5], o[3] = p[4], o[4] = p[6], o[5] = p[7], o[6] = p[5], o[7] = p[7], o[8] = p[8];
  }
  if (cross9) {
    double *o = cross9 + 9 * (size_t)i;
    o[0] = 0, o[1] = -p[2], o[2] = p[1], o[3] = p[2], o[4] = 0, o[5] = -p[0], o[6] = -p[1], o[7] = p[0], o[8] = 0;
  }
}

int esikf_lio_fetch_point_cov(esikf_ctx *ctx, double *body_cov9, double *cross_mat9) {
  if (!ctx) return ESIKF_ERR_ARG;
  if (ctx->scan_fresh) return fail(ctx, ESIKF_ERR_STATE, "fetch_point_cov before lio_run");
  CK(cudaSetDevice(ctx->device));
  const int n = ctx->n_pts;
  if (n == 0) return ESIKF_OK;
  DevBuf<double> &tmp = ctx->point_cov_tmp;  // context-owned scratch: no allocation per tick once it has grown
  CK(tmp.reserve((size_t)n * 18));
  expand_point_cov_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->pre.p, ctx->pre_stride, n, body_cov9 ? tmp.p : nullptr, cross_mat9 ? tmp.p + 9 * (size_t)n : nullptr);
  ctx->launches++;
  if (body_cov9) CK(cudaMemcpyAsync(body_cov9, tmp.p, (size_t)n * 9 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (cross_mat9) CK(cudaMemcpyAsync(cross_mat9, tmp.p + 9 * (size_t)n, (size_t)n * 9 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return ESIKF_OK;
}

// ---------------------------------------------------------------------------------------------------------------- VIO
int esikf_vio_set_camera(esikf_ctx *ctx, const esikf_camera *cam, const esikf_vio_cfg *cfg) {
  if (!ctx || !cam || !cfg) return fail(ctx, ESIKF_ERR_ARG, "vio_set_camera: null argument");
  if (cam->model < 0 || cam->model > 1 || cam->width <= 0 || cam->height <= 0) return fail(ctx, ESIKF_ERR_ARG, "vio_set_camera: bad camera");
  if (cfg->patch_pyrimid_level < 1 || cfg->patch_pyrimid_level > 8 || cfg->max_iterations < 1 || cfg->max_iterations > 8 || !(cfg->img_point_cov > 0))
    return fail(ctx, ESIKF_ERR_ARG, "vio_set_camera: bad vio cfg");
  ctx->cam = *cam;
  ctx->vio_cfg = *cfg;
  ctx->have_cam = true;
  return ESIKF_OK;
}

int esikf_vio_set_image(esikf_ctx *ctx, const uint8_t *img, int32_t width, int32_t height) {
  if (!ctx || !img || width <= 0 || height <= 0) return fail(ctx, ESIKF_ERR_ARG, "vio_set_image: bad argument");
  if (!ctx->have_cam) return fail(ctx, ESIKF_ERR_STATE, "vio_set_image before vio_set_camera");
  if (width != ctx->cam.width || height != ctx->cam.height) return fail(ctx, ESIKF_ERR_ARG, "vio_set_image: image is %dx%d, camera %dx%d", width, height, ctx->cam.width, ctx->cam.height);
  CK(cudaSetDevice(ctx->device));
  CK(ctx->img.upload(img, (size_t)width * height, (size_t)width * height + 64, ctx->stream));
  ctx->img_w = width, ctx->img_h = height;
  return ESIKF_OK;
}

// The kernels shift by the tap stride 1 << (level + search_level) and index the per-stride tensor maps with it: search
// levels must lie in [0, 8]. `name_patch` adds the patch number to the message.
static int check_search_levels(esikf_ctx *ctx, const char *what, const int32_t *levels, int n, bool name_patch) {
  for (int i = 0; i < n; i++)
    if (levels[i] < 0 || levels[i] > 8)
      return name_patch ? fail(ctx, ESIKF_ERR_ARG, "%s: search level %d of patch %d", what, levels[i], i) : fail(ctx, ESIKF_ERR_ARG, "%s: search level %d", what, levels[i]);
  return ESIKF_OK;
}
static int check_ref_indices(esikf_ctx *ctx, const char *what, const int32_t *ref_img_index, int n) {
  for (int i = 0; i < n; i++)
    if (ref_img_index[i] < 0 || ref_img_index[i] >= (int)ctx->ref_imgs.size()) return fail(ctx, ESIKF_ERR_ARG, "%s: ref image index %d", what, ref_img_index[i]);
  return ESIKF_OK;
}

int esikf_vio_set_patches(esikf_ctx *ctx, const double *pos, const float *warp_patch, const int32_t *search_levels, const double *inv_expo_list, int32_t n) {
  if (!ctx || n < 0 || (n > 0 && (!pos || !warp_patch || !search_levels || !inv_expo_list))) return fail(ctx, ESIKF_ERR_ARG, "vio_set_patches: bad argument");
  if (!ctx->have_cam) return fail(ctx, ESIKF_ERR_STATE, "vio_set_patches before vio_set_camera");
  // checked before anything is uploaded so the installed patches stay as they were
  int rc = check_search_levels(ctx, "vio_set_patches", search_levels, n, true);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  const size_t L = ctx->vio_cfg.patch_pyrimid_level;
  cudaStream_t st = ctx->stream;
  CK(ctx->vis_pos.upload(pos, (size_t)n * 3, (size_t)n * 3 + 4, st));
  CK(ctx->warp_patch.upload(warp_patch, n * 64 * L, n * 64 * L + 64, st));
  CK(ctx->search_levels.upload(search_levels, n, n + 1, st));
  CK(ctx->inv_expo.upload(inv_expo_list, n, n + 1, st));
  CK(ctx->errors.reserve(n + 1));
  ctx->n_patches = n;
  return ESIKF_OK;
}

static void vio_consts(const esikf_ctx *ctx, double Rci[9], double Pci[3], double Jdp_dR[9]) {
  // vio.cpp:29-33, 57-65: Rli = extR^T, Pli = -extR^T extT, Rci = Rcl Rli, Pci = Rcl Pli + Pcl, Pic = -Rci^T Pci, Jdp_dR = -Rci [Pic]x
  const esikf_extrinsics &e = ctx->ext;
  double Rli[9], Pli[3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) Rli[3 * r + c] = e.extR[3 * c + r];
  for (int r = 0; r < 3; r++) Pli[r] = -(Rli[3 * r] * e.extT[0] + Rli[3 * r + 1] * e.extT[1] + Rli[3 * r + 2] * e.extT[2]);
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) Rci[3 * r + c] = e.Rcl[3 * r] * Rli[c] + e.Rcl[3 * r + 1] * Rli[3 + c] + e.Rcl[3 * r + 2] * Rli[6 + c];
  for (int r = 0; r < 3; r++) Pci[r] = e.Rcl[3 * r] * Pli[0] + e.Rcl[3 * r + 1] * Pli[1] + e.Rcl[3 * r + 2] * Pli[2] + e.Pcl[r];
  double Pic[3];
  for (int r = 0; r < 3; r++) Pic[r] = -(Rci[r] * Pci[0] + Rci[3 + r] * Pci[1] + Rci[6 + r] * Pci[2]);
  const double tmp[9] = {0.0, -Pic[2], Pic[1], Pic[2], 0.0, -Pic[0], -Pic[1], Pic[0], 0.0};
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) Jdp_dR[3 * r + c] = -(Rci[3 * r] * tmp[c] + Rci[3 * r + 1] * tmp[3 + c] + Rci[3 * r + 2] * tmp[6 + c]);
}
static void cam_dev(const esikf_ctx *ctx, CamDev &c) {
  c.model = ctx->cam.model, c.width = ctx->cam.width, c.height = ctx->cam.height;
  c.fx = ctx->cam.fx, c.fy = ctx->cam.fy, c.cx = ctx->cam.cx, c.cy = ctx->cam.cy;
  for (int i = 0; i < 5; i++) c.d[i] = ctx->cam.d[i];
}
static void vio_fill_args(esikf_ctx *ctx, VioKernelArgs &ka, double *state_ptr) {
  memset(&ka, 0, sizeof(ka));
  ka.img = ctx->img.p;
  cam_dev(ctx, ka.cam);
  ka.pos = ctx->vis_pos.p, ka.warp_patch = ctx->warp_patch.p, ka.search_levels = ctx->search_levels.p, ka.inv_expo_list = ctx->inv_expo.p;
  shard_of(ctx->n_patches, ctx->rank, ctx->nranks, ka.begin, ka.count);
  ka.levels = ctx->vio_cfg.patch_pyrimid_level;
  ka.exposure_en = ctx->vio_cfg.exposure_estimate_en;
  ka.state = state_ptr;
  vio_consts(ctx, ka.Rci, ka.Pci, ka.Jdp_dR);
  ka.errors = ctx->errors.p, ka.partials = ctx->partials.p, ka.info = ctx->info.p, ka.ctrl = &ctx->ctl.p->ctrl;
  ka.partial_stride = ctx->partial_blocks;
}
static int vio_grid(const esikf_ctx *ctx, int count) {
  int g = (count + VIO_WARPS - 1) / VIO_WARPS;  // one patch per warp while the patches last
  if (g > ctx->partial_blocks) g = ctx->partial_blocks;
  return g < 1 ? 1 : g;
}

// Tiled tensor maps of the level-0 u8 image, one per tap stride 1 << l (see VioTma). Encoded through the driver entry
// point (no link-time dependency on libcuda). Images whose row pitch is not a multiple of 16 bytes cannot be described:
// the variant then stays on the per-lane loads (enabled = 0).
static int vio_encode_tma(esikf_ctx *ctx) {
  if (ctx->tma_img == ctx->img.p && ctx->tma_w == ctx->img_w && ctx->tma_h == ctx->img_h) return ESIKF_OK;
  memset(&ctx->tma, 0, sizeof(ctx->tma));
  ctx->tma_img = ctx->img.p, ctx->tma_w = ctx->img_w, ctx->tma_h = ctx->img_h;
  if (ctx->img_w % 16 != 0 || ((uintptr_t)ctx->img.p & 15)) return ESIKF_OK;
  typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  void *fn = nullptr;
  cudaDriverEntryPointQueryResult qr;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess || !fn)
    return fail(ctx, ESIKF_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  static_assert(sizeof(CUtensorMap) == 128, "descriptor size");
  for (int l = 0; l <= VIO_TMA_MAXLVL; l++) {
    const cuuint64_t dims[2] = {(cuuint64_t)ctx->img_w, (cuuint64_t)ctx->img_h};
    const cuuint64_t strides[1] = {(cuuint64_t)ctx->img_w};  // bytes between rows
    const cuuint32_t box[2] = {VIO_TMA_INNER(l), 11u << l};
    const cuuint32_t estr[2] = {1u, 1u << l};
    CUresult r = ((encode_fn)fn)(reinterpret_cast<CUtensorMap *>(ctx->tma.map[l]), CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void *)ctx->img.p, dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, ESIKF_ERR_CUDA, "cuTensorMapEncodeTiled (tap stride %d) failed: %d", 1 << l, (int)r);
  }
  ctx->tma.enabled = 1;
  return ESIKF_OK;
}

int esikf_vio_run(esikf_ctx *ctx, const double *state_in, const double *state_prop) {
  if (!ctx || !state_in || !state_prop) return fail(ctx, ESIKF_ERR_ARG, "vio_run: null argument");
  if (!ctx->have_cam || !ctx->have_ext) return fail(ctx, ESIKF_ERR_STATE, "vio_run before vio_set_camera / set_extrinsics");
  if (ctx->img_w == 0) return fail(ctx, ESIKF_ERR_STATE, "vio_run before vio_set_image");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  {
    int rc = upload_states(ctx, state_in, state_prop);
    if (rc) return rc;
  }
  const bool inverse = ctx->vio_cfg.inverse_composition_en != 0;
  if (inverse && ctx->n_patches > 0) {
    if (ctx->n_inv_refs != ctx->n_patches) return fail(ctx, ESIKF_ERR_STATE, "vio_run: inverse_composition_en needs esikf_vio_set_inverse_refs for the %d patches (have %d)", ctx->n_patches, ctx->n_inv_refs);
    if (ctx->ref_w != ctx->cam.width || ctx->ref_h != ctx->cam.height) return fail(ctx, ESIKF_ERR_STATE, "vio_run: reference images must have the camera's size");
  }
  const bool fused_vio = ctx->n_patches > 0 && persistent_ok(ctx, ctx->coop_vio);
  if (!fused_vio) {
    CK(cudaMemsetAsync(&ctx->ctl.p->ctrl, 0, sizeof(Ctrl), st));
    CK(cudaMemsetAsync(&ctx->ctl.p->vio_stats, 0, sizeof(esikf_vio_stats), st));
  }
  if (ctx->n_patches == 0) return ESIKF_OK;  // total_points == 0: early return (vio.cpp:786)
  VioKernelArgs ka;
  vio_fill_args(ctx, ka, ctx->state);
  SolveArgs sa = solve_args(ctx, ctx->state, ctx->vio_cfg.max_iterations);
  sa.vio_stats = &ctx->ctl.p->vio_stats;
  sa.old_state = ctx->old_state.p, sa.G = ctx->G.p, sa.img_point_cov = ctx->vio_cfg.img_point_cov;
  const int grid = vio_grid(ctx, ka.count);
  VioInvArgs iv;
  memset(&iv, 0, sizeof(iv));
  if (inverse) {
    CK(ctx->H_sub_inv.reserve((size_t)ka.count * 64 * 6 + 8));
    iv.ref_imgs = ctx->ref_img_ptrs.p, iv.ref_idx = ctx->inv_ref_idx.p, iv.ref_px = ctx->inv_ref_px.p, iv.ref_f = ctx->inv_ref_f.p;
    iv.ref_R = ctx->inv_ref_R.p, iv.ref_pos = ctx->inv_ref_pos.p, iv.H_sub_inv = ctx->H_sub_inv.p;
    iv.ref_w = ctx->ref_w, iv.ref_h = ctx->ref_h, iv.fx = ctx->cam.fx, iv.fy = ctx->cam.fy;
  }
  if (fused_vio) {
    VioTma tma_off;
    tma_off.enabled = 0;
    VioTma *tma = &tma_off;
    if (ctx->tuning & ESIKF_TUNE_VIO_TMA) {
      int rc = vio_encode_tma(ctx);
      if (rc) return rc;
      tma = &ctx->tma;
    }
    const void *solo = inverse ? (const void *)vio_update_kernel<false, true> : (const void *)vio_update_kernel<false, false>;
    const void *peers = inverse ? (const void *)vio_update_kernel<true, true> : (const void *)vio_update_kernel<true, false>;
    return launch_persistent(ctx, "vio_update_kernel", solo, peers, grid, VIO_THREADS, VIO_PERSIST_SMEM, 64, 512, &ka, &sa, &iv, tma, ctx->vio_timed);
  }
  ctx->vio_timed = ctx->timing;
  ctx->vio_slots = ctx->vio_cfg.patch_pyrimid_level * ctx->vio_cfg.max_iterations;
  int slot = 0;
  for (int level = ctx->vio_cfg.patch_pyrimid_level - 1; level >= 0; level--) {
    if (inverse) {  // has_ref_patch_cache = false at every level (vio.cpp:794): H_sub_inv of this level's tap stride
      vio_inverse_precompute_kernel<<<(ka.count + 7) / 8, 256, 0, st>>>(ka, iv, level);
      ctx->launches++;
    }
    for (int it = 0; it < ctx->vio_cfg.max_iterations; it++, slot++) {
      ka.level = level, ka.slot_iter = it;
      cudaEvent_t *e = ctx->timing ? timing_events(ctx, EV_VIO_BASE, slot) : nullptr;
      if (e) cudaEventRecord(e[0], st);
      if (inverse)
        vio_inverse_patch_kernel<<<grid, VIO_THREADS, sizeof(VioSmem), st>>>(ka, iv);
      else
        vio_patch_kernel<<<grid, VIO_THREADS, sizeof(VioSmem), st>>>(ka);
      if (e) cudaEventRecord(e[1], st);
      int rc = allreduce_info(ctx);
      if (rc) return rc;
      sa.level = level, sa.slot_iter = it, sa.last_slot = (level == 0 && it == ctx->vio_cfg.max_iterations - 1);
      vio_solve_kernel<<<1, SOLVE_THREADS, 0, st>>>(sa);
      if (e) cudaEventRecord(e[2], st);
      ctx->launches += 2;
    }
  }
  CK(cudaGetLastError());
  return ESIKF_OK;
}

int esikf_vio_fetch(esikf_ctx *ctx, double *state_out, esikf_vio_stats *stats, float *errors) {
  if (!ctx) return ESIKF_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  if (state_out) CK(cudaMemcpyAsync(state_out, ctx->state, S_N * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (stats) CK(cudaMemcpyAsync(stats, &ctx->ctl.p->vio_stats, sizeof(esikf_vio_stats), cudaMemcpyDeviceToHost, st));
  if (errors && ctx->n_patches) CK(cudaMemcpyAsync(errors, ctx->errors.p, (size_t)ctx->n_patches * sizeof(float), cudaMemcpyDeviceToHost, st));
  return finish_fetch(ctx);
}

int esikf_vio_update(esikf_ctx *ctx, const uint8_t *img, int32_t width, int32_t height, const double *pos, const float *warp_patch,
                     const int32_t *search_levels, const double *inv_expo_list, int32_t n, const double *state_in, const double *state_prop,
                     double *state_out, esikf_vio_stats *stats, float *errors) {
  int rc = esikf_vio_set_image(ctx, img, width, height);
  if (rc) return rc;
  rc = esikf_vio_set_patches(ctx, pos, warp_patch, search_levels, inv_expo_list, n);
  if (rc) return rc;
  rc = esikf_vio_run(ctx, state_in, state_prop);
  if (rc) return rc;
  return esikf_vio_fetch(ctx, state_out, stats, errors);
}

// ---------------------------------------------------------------------------------------------------------------- patch producers
int esikf_vio_get_image_patch(esikf_ctx *ctx, const double *pc, int32_t n, int32_t level, float *patch_out) {
  if (!ctx || n < 0 || level < 0 || level > 12 || (n > 0 && (!pc || !patch_out))) return fail(ctx, ESIKF_ERR_ARG, "get_image_patch: bad argument");
  if (ctx->img_w == 0) return fail(ctx, ESIKF_ERR_STATE, "get_image_patch before vio_set_image");
  if (n == 0) return ESIKF_OK;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CK(ctx->pc_buf.upload(pc, (size_t)n * 2, (size_t)n * 2, st));
  CK(ctx->patch_buf.reserve((size_t)n * 64));
  image_patch_kernel<<<(n * 64 + 255) / 256, 256, 0, st>>>(ctx->img.p, ctx->img_w, ctx->img_h, ctx->pc_buf.p, n, level, ctx->patch_buf.p);
  ctx->launches++;
  CK(cudaMemcpyAsync(patch_out, ctx->patch_buf.p, (size_t)n * 64 * sizeof(float), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return ESIKF_OK;
}

int esikf_vio_set_ref_images(esikf_ctx *ctx, const uint8_t *const *imgs, int32_t n_imgs, int32_t width, int32_t height) {
  if (!ctx || n_imgs < 0 || width <= 0 || height <= 0 || (n_imgs > 0 && !imgs)) return fail(ctx, ESIKF_ERR_ARG, "set_ref_images: bad argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->ref_imgs.clear();
  ctx->n_inv_refs = 0;  // the inverse-compositional reference indices pointed into the images just released
  std::vector<const uint8_t *> ptrs;
  for (int i = 0; i < n_imgs; i++) {
    DevBuf<uint8_t> d;
    CK(d.upload(imgs[i], (size_t)width * height, (size_t)width * height + 64, ctx->stream));
    ptrs.push_back(d.p);
    ctx->ref_imgs.push_back(std::move(d));
  }
  CK(ctx->ref_img_ptrs.upload(ptrs.data(), n_imgs, n_imgs + 1, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->ref_w = width, ctx->ref_h = height;
  return ESIKF_OK;
}

int esikf_vio_warp_patches(esikf_ctx *ctx, int32_t n, const int32_t *ref_img_index, const double *px_ref, const double *pos_w, const double *normal_w,
                           const double *T_ref_w, const double *T_cur_w, double *A_cur_ref_out, int32_t *search_level_out, float *warp_patch_out,
                           int32_t keep_on_device) {
  if (!ctx || n < 0 || (n > 0 && (!ref_img_index || !px_ref || !pos_w || !normal_w || !T_ref_w || !T_cur_w)))
    return fail(ctx, ESIKF_ERR_ARG, "warp_patches: bad argument");
  if (!ctx->have_cam) return fail(ctx, ESIKF_ERR_STATE, "warp_patches before vio_set_camera");
  if (ctx->ref_imgs.empty()) return fail(ctx, ESIKF_ERR_STATE, "warp_patches before set_ref_images");
  int rc = check_ref_indices(ctx, "warp_patches", ref_img_index, n);
  if (rc) return rc;
  if (n == 0) return ESIKF_OK;
  CK(cudaSetDevice(ctx->device));
  const int L = ctx->vio_cfg.patch_pyrimid_level;
  cudaStream_t st = ctx->stream;
  CK(ctx->ref_idx.upload(ref_img_index, n, n, st));
  CK(ctx->px_ref.upload(px_ref, (size_t)n * 2, (size_t)n * 2, st));
  CK(ctx->pos_w.upload(pos_w, (size_t)n * 3, (size_t)n * 3, st));
  CK(ctx->normal_w.upload(normal_w, (size_t)n * 3, (size_t)n * 3, st));
  CK(ctx->T_ref.upload(T_ref_w, (size_t)n * 12, (size_t)n * 12, st));
  CK(ctx->T_cur.upload(T_cur_w, 12, 12, st));
  CK(ctx->A_cur_ref.reserve((size_t)n * 4));
  CK(ctx->search_levels.reserve(n + 1));
  CK(ctx->warp_patch.reserve((size_t)n * 64 * L + 64));
  CamDev cam;
  cam_dev(ctx, cam);
  warp_matrix_kernel<<<(n + 127) / 128, 128, 0, st>>>(cam, n, ctx->px_ref.p, ctx->pos_w.p, ctx->normal_w.p, ctx->T_ref.p, ctx->T_cur.p, ctx->A_cur_ref.p,
                                                     ctx->search_levels.p);
  CK(cudaMemsetAsync(ctx->warp_patch.p, 0, (size_t)n * 64 * L * sizeof(float), st));
  warp_affine_kernel<<<(n * L * 64 + 255) / 256, 256, 0, st>>>(ctx->ref_img_ptrs.p, ctx->ref_idx.p, ctx->ref_w, ctx->ref_h, n, L, ctx->A_cur_ref.p,
                                                              ctx->px_ref.p, ctx->search_levels.p, ctx->warp_patch.p);
  ctx->launches += 2;
  if (A_cur_ref_out) CK(cudaMemcpyAsync(A_cur_ref_out, ctx->A_cur_ref.p, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (search_level_out) CK(cudaMemcpyAsync(search_level_out, ctx->search_levels.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (warp_patch_out) CK(cudaMemcpyAsync(warp_patch_out, ctx->warp_patch.p, (size_t)n * 64 * L * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (keep_on_device) {
    // install as the visual sub-map of the coming update: pos = pos_w, inv_expo filled by the caller through set_patches otherwise
    CK(ctx->vis_pos.reserve((size_t)n * 3 + 4));
    CK(ctx->errors.reserve(n + 1));
    CK(cudaMemcpyAsync(ctx->vis_pos.p, ctx->pos_w.p, (size_t)n * 3 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    std::vector<double> ones(n, 1.0);
    CK(ctx->inv_expo.upload(ones.data(), n, n + 1, st));
    CK(cudaStreamSynchronize(st));
    ctx->n_patches = n;
  }
  CK(cudaStreamSynchronize(st));
  return ESIKF_OK;
}

int esikf_vio_set_inverse_refs(esikf_ctx *ctx, int32_t n, const int32_t *ref_img_index, const double *ref_px, const double *ref_f, const double *ref_R,
                               const double *ref_pos) {
  if (!ctx || n < 0 || (n > 0 && (!ref_img_index || !ref_px || !ref_f || !ref_R || !ref_pos))) return fail(ctx, ESIKF_ERR_ARG, "set_inverse_refs: bad argument");
  if (ctx->ref_imgs.empty() && n > 0) return fail(ctx, ESIKF_ERR_STATE, "set_inverse_refs before set_ref_images");
  int rc = check_ref_indices(ctx, "set_inverse_refs", ref_img_index, n);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CK(ctx->inv_ref_idx.upload(ref_img_index, n, n + 1, st));
  CK(ctx->inv_ref_px.upload(ref_px, (size_t)n * 2, (size_t)n * 2 + 2, st));
  CK(ctx->inv_ref_f.upload(ref_f, (size_t)n * 3, (size_t)n * 3 + 3, st));
  CK(ctx->inv_ref_R.upload(ref_R, (size_t)n * 9, (size_t)n * 9 + 9, st));
  CK(ctx->inv_ref_pos.upload(ref_pos, (size_t)n * 3, (size_t)n * 3 + 3, st));
  if (n > 0) CK(cudaStreamSynchronize(st));  // the caller's arrays may go away
  ctx->n_inv_refs = n;
  return ESIKF_OK;
}

int esikf_vio_warp_affine(esikf_ctx *ctx, int32_t n, const int32_t *ref_img_index, const double *px_ref, const double *A_cur_ref,
                          const int32_t *search_level, float *warp_patch_out) {
  if (!ctx || n < 0 || (n > 0 && (!ref_img_index || !px_ref || !A_cur_ref || !search_level || !warp_patch_out)))
    return fail(ctx, ESIKF_ERR_ARG, "warp_affine: bad argument");
  if (!ctx->have_cam) return fail(ctx, ESIKF_ERR_STATE, "warp_affine before vio_set_camera");
  if (ctx->ref_imgs.empty()) return fail(ctx, ESIKF_ERR_STATE, "warp_affine before set_ref_images");
  int rc = check_ref_indices(ctx, "warp_affine", ref_img_index, n);
  if (!rc) rc = check_search_levels(ctx, "warp_affine", search_level, n, false);
  if (rc) return rc;
  if (n == 0) return ESIKF_OK;
  CK(cudaSetDevice(ctx->device));
  const int L = ctx->vio_cfg.patch_pyrimid_level;
  cudaStream_t st = ctx->stream;
  CK(ctx->ref_idx.upload(ref_img_index, n, n, st));
  CK(ctx->px_ref.upload(px_ref, (size_t)n * 2, (size_t)n * 2, st));
  CK(ctx->A_cur_ref.upload(A_cur_ref, (size_t)n * 4, (size_t)n * 4, st));
  CK(ctx->warp_levels.upload(search_level, n, n + 1, st));
  CK(ctx->warp_out.reserve((size_t)n * 64 * L + 64));
  // separate scratch: the patches / search levels installed by set_patches (or warp_patches with keep_on_device) stay untouched
  CK(cudaMemsetAsync(ctx->warp_out.p, 0, (size_t)n * 64 * L * sizeof(float), st));
  warp_affine_kernel<<<(n * L * 64 + 255) / 256, 256, 0, st>>>(ctx->ref_img_ptrs.p, ctx->ref_idx.p, ctx->ref_w, ctx->ref_h, n, L, ctx->A_cur_ref.p,
                                                              ctx->px_ref.p, ctx->warp_levels.p, ctx->warp_out.p);
  ctx->launches += 1;
  CK(cudaMemcpyAsync(warp_patch_out, ctx->warp_out.p, (size_t)n * 64 * L * sizeof(float), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  return ESIKF_OK;
}

// ---------------------------------------------------------------------------------------------------------------- multi-GPU
int esikf_comm_unique_id(char out[128]) {
  if (!out) return ESIKF_ERR_ARG;
  if (!g_nccl.load()) return ESIKF_ERR_COMM;
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != 0) return ESIKF_ERR_COMM;
  memcpy(out, id.internal, 128);
  return ESIKF_OK;
}
int esikf_comm_init(esikf_ctx *ctx, int32_t rank, int32_t nranks, const char unique_id[128]) {
  if (!ctx || nranks < 1 || rank < 0 || rank >= nranks || !unique_id) return fail(ctx, ESIKF_ERR_ARG, "comm_init: bad argument");
  if (nranks == 1) {
    ctx->rank = 0, ctx->nranks = 1;
    return ESIKF_OK;
  }
  if (!g_nccl.load()) return fail(ctx, ESIKF_ERR_COMM, "libnccl.so.2 not found");
  CK(cudaSetDevice(ctx->device));
  ncclUniqueId id;
  memcpy(id.internal, unique_id, 128);
  int r = g_nccl.CommInitRank(&ctx->comm, nranks, id, rank);
  if (r != 0) return fail(ctx, ESIKF_ERR_COMM, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  ctx->rank = rank, ctx->nranks = nranks;
  return ESIKF_OK;
}
int esikf_peer_export(esikf_ctx *ctx, char out[64]) {
  if (!ctx || !out) return ESIKF_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  if (!ctx->mailbox) {
    const size_t words = (size_t)2 * PEER_MAX_RANKS * PEER_SLOT_WORDS + 2;  // + the exchange counter
    CK(cudaMalloc(&ctx->mailbox, words * sizeof(unsigned long long)));
    CK(cudaMemset(ctx->mailbox, 0, words * sizeof(unsigned long long)));  // tag 0 is never sent
    ctx->peer_seq_dev = reinterpret_cast<unsigned int *>(ctx->mailbox + (size_t)2 * PEER_MAX_RANKS * PEER_SLOT_WORDS);
  }
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, ctx->mailbox));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(out, &h, 64);
  return ESIKF_OK;
}
int esikf_peer_attach(esikf_ctx *ctx, int32_t rank, int32_t nranks, const char *handles) {
  if (!ctx || !handles || nranks < 1 || nranks > PEER_MAX_RANKS || rank < 0 || rank >= nranks) return fail(ctx, ESIKF_ERR_ARG, "peer_attach: bad argument (1..8 ranks)");
  if (!ctx->mailbox) return fail(ctx, ESIKF_ERR_STATE, "peer_attach before peer_export");
  CK(cudaSetDevice(ctx->device));
  ctx->peer_ptrs.assign(nranks, nullptr);
  for (int r = 0; r < nranks; r++) {
    if (r == rank) {
      ctx->peer_ptrs[r] = ctx->mailbox;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + 64 * (size_t)r, 64);
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(ctx, ESIKF_ERR_COMM, "cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
    ctx->peer_ptrs[r] = (unsigned long long *)p;
  }
  CK(ctx->peer_ptrs_dev.reserve(nranks));
  CK(cudaMemcpy(ctx->peer_ptrs_dev.p, ctx->peer_ptrs.data(), nranks * sizeof(unsigned long long *), cudaMemcpyHostToDevice));
  // mailbox and exchange counter were zeroed at export time (before the host-side all-gather): a peer may already be writing
  ctx->rank = rank, ctx->nranks = nranks, ctx->p2p = true;
  return ESIKF_OK;
}
int esikf_shard_range(int32_t n, int32_t rank, int32_t nranks, int32_t *begin, int32_t *count) {
  if (n < 0 || nranks < 1 || rank < 0 || rank >= nranks || !begin || !count) return ESIKF_ERR_ARG;
  int b, c;
  shard_of(n, rank, nranks, b, c);
  *begin = b, *count = c;
  return ESIKF_OK;
}
int esikf_comm_rank(const esikf_ctx *ctx, int32_t *rank, int32_t *nranks) {
  if (!ctx) return ESIKF_ERR_ARG;
  if (rank) *rank = ctx->rank;
  if (nranks) *nranks = ctx->nranks;
  return ESIKF_OK;
}

// ---------------------------------------------------------------------------------------------------------------- measurement
int esikf_profile_kernel(esikf_ctx *ctx, int32_t which, int32_t arg, int32_t reps, int32_t flush_l2, float *avg_ms) {
  if (!ctx || !avg_ms || reps < 1) return fail(ctx, ESIKF_ERR_ARG, "profile_kernel: bad argument");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t flush_bytes = 256u << 20;
  if (flush_l2) CK(ctx->flush.reserve(flush_bytes));
  // work on a scratch copy of the resident state so the measured launches never disturb an update in flight
  Ctrl *ctrl = &ctx->ctl.p->ctrl;
  CK(cudaMemcpyAsync(ctx->scratch_state.p, ctx->state, S_N * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemsetAsync(ctrl, 0, sizeof(Ctrl), st));
  cudaEvent_t e0 = ctx->prof_ev[0], e1 = ctx->prof_ev[1];
  double total = 0.0;
  LioKernelArgs la;
  VioKernelArgs va;
  SolveArgs sa{};
  int grid = 1;
  if (which == 0 || which == 1 || which == 3) {
    if (!ctx->have_map || ctx->n_pts == 0 || ctx->scan_fresh) return fail(ctx, ESIKF_ERR_STATE, "profile_kernel: no resident LIO frame (run lio once)");
    lio_fill_args(ctx, la, ctx->scratch_state.p);
    grid = lio_grid(ctx, la.count);
    sa = solve_args(ctx, ctx->scratch_state.p, 1 << 20);
  } else if (which == 2) {
    if (ctx->n_patches == 0 || ctx->img_w == 0) return fail(ctx, ESIKF_ERR_STATE, "profile_kernel: no resident VIO frame");
    vio_fill_args(ctx, va, ctx->scratch_state.p);
    va.level = arg, va.slot_iter = 0;
    grid = vio_grid(ctx, va.count);
  } else {
    return fail(ctx, ESIKF_ERR_ARG, "profile_kernel: which=%d", which);
  }
  for (int r = 0; r < reps + 3; r++) {  // 3 warm-up launches
    if (flush_l2) CK(cudaMemsetAsync(ctx->flush.p, r & 0xff, flush_bytes, st));
    if (which == 1) {
      CK(cudaMemcpyAsync(ctx->scratch_state.p, ctx->state, S_N * sizeof(double), cudaMemcpyDeviceToDevice, st));
      CK(cudaMemsetAsync(ctrl, 0, sizeof(Ctrl), st));
    }
    CK(cudaEventRecord(e0, st));
    if (which == 0) lio_residual_kernel<<<grid, LIO_THREADS, sizeof(LioSmem), st>>>(la);
    else if (which == 1) lio_solve_kernel<<<1, SOLVE_THREADS, 0, st>>>(sa);
    else if (which == 2) vio_patch_kernel<<<grid, VIO_THREADS, sizeof(VioSmem), st>>>(va);
    else lio_precompute_kernel<<<(ctx->n_pts + 255) / 256, 256, 0, st>>>(ctx->pts.p, ctx->n_pts, ctx->pre.p, ctx->pre_stride, ctx->ext_dev.p, (float)ctx->lio_cfg.dept_err,
                                                                       (float)ctx->lio_cfg.beam_err);
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    ctx->launches++;
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    if (r >= 3) total += ms;
  }
  CK(cudaGetLastError());
  *avg_ms = (float)(total / reps);
  return ESIKF_OK;
}

int esikf_set_phase_stamps(esikf_ctx *ctx, int32_t enable) {
  if (!ctx) return ESIKF_ERR_ARG;
  ctx->want_stamps = enable != 0;
  return ESIKF_OK;
}
int esikf_get_phase_stamps(esikf_ctx *ctx, uint64_t *out /* 800 */) {
  if (!ctx || !out) return ESIKF_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(out, ctx->stamps.p, 800 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return ESIKF_OK;
}

int esikf_set_kernel_timing(esikf_ctx *ctx, int32_t enable) {
  if (!ctx) return ESIKF_ERR_ARG;
  ctx->timing = enable != 0;
  return ESIKF_OK;
}

int esikf_get_kernel_timing(esikf_ctx *ctx, float *lio_residual_ms, float *lio_solve_ms, float *vio_patch_ms, float *vio_solve_ms) {
  if (!ctx) return ESIKF_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int pass = 0; pass < 2; pass++) {
    const bool timed = pass == 0 ? ctx->lio_timed : ctx->vio_timed;
    const int slots = pass == 0 ? ctx->lio_slots : ctx->vio_slots, base = pass == 0 ? EV_LIO_BASE : EV_VIO_BASE, cap = pass == 0 ? 8 : 64;
    float *a = pass == 0 ? lio_residual_ms : vio_patch_ms, *b = pass == 0 ? lio_solve_ms : vio_solve_ms;
    for (int i = 0; i < cap; i++) {
      if (a) a[i] = 0.f;
      if (b) b[i] = 0.f;
    }
    if (!timed) continue;
    for (int i = 0; i < slots && i < cap; i++) {
      cudaEvent_t *e = &ctx->ev[(size_t)(base + i) * 3];
      float ms = 0.f;
      if (a && cudaEventElapsedTime(&ms, e[0], e[1]) == cudaSuccess) a[i] = ms;
      if (b && cudaEventElapsedTime(&ms, e[1], e[2]) == cudaSuccess) b[i] = ms;
    }
  }
  return ESIKF_OK;
}

}  // extern "C"
