// Persistent update kernels of the B200 ESIKF update (sm_100a): the WHOLE iteration loop of one LIO / VIO update in a
// single cooperative launch, so a tick costs one launch instead of 2 x iterations, the state never leaves the chip between
// iterations and no kernel boundary separates the residual build from the gain solve.
//
//   lio_update_kernel : VoxelMapManager::StateEstimation's loop          (reference src/voxel_map.cpp:372-500)
//   vio_update_kernel : VIOManager::computeJacobianAndUpdateEKF's loops   (src/vio.cpp:784-802, 1520-1688)
//
// Every CTA (one per SM, co-resident) keeps its own copy of P, the current / prior pose and the loop control in shared
// memory for the whole update. Per iteration: build the residual / Jacobian rows of the CTA's slice and contract them on
// the fp64 tensor-core path -> write the CTA's compact partial vector (double-buffered by iteration parity) -> ONE grid
// barrier (state_propagat (-) state is evaluated inside the wait) -> every CTA sums the partial columns in the same fixed
// order and runs the same m x m gain solve and boxplus — same instructions on the same inputs, so all copies stay
// bit-identical. Only the LAST CTA writes results and diagnostics (its slice is never the largest, so the
// stores stay off the critical path of the grid). With peer GPUs attached (PEER) CTA 0 additionally pushes the
// rank's vector into every rank's NVLink mailbox and every CTA adds the rank-ordered sum pulled from the local one.
#include "esikf_dev.cuh"

namespace esikf {

// Optional phase timestamps (ns, %globaltimer) written by CTA 0 / thread 0 — measurement only.
__device__ __forceinline__ void stamp(unsigned long long *stamps, int &k) {
  if (stamps && blockIdx.x == 0 && threadIdx.x == 0) stamps[k] = globaltimer_ns();
  k++;
}

// Every wait inside the persistent kernels (grid barrier, peer mailbox) is bounded: a rank that never arrives must not
// hang the other seven. On expiry the waiter raises Ctrl::comm_error (host: ESIKF_ERR_COMM at fetch) and stops waiting for
// the rest of the launch; the numbers of that update are invalid but the kernel terminates.
#define ESIKF_WAIT_NS 2000000000ull
struct WaitGuard {
  int *error_flag;  // Ctrl::comm_error in global memory
  bool dead;
};
__device__ __forceinline__ bool wait_expired(WaitGuard &w, unsigned long long t0, unsigned &spins) {
  if ((++spins & 1023u) != 0) return false;
  if (globaltimer_ns() - t0 < ESIKF_WAIT_NS) return false;
  w.dead = true;
  *reinterpret_cast<volatile int *>(w.error_flag) = 1;
  return true;
}

// ---------------------------------------------------------------------------------------------------------------------
// In-kernel all-reduce of the compact information vector over NVLink peer memory (one process per GPU, mailboxes
// exchanged with CUDA IPC), low-latency flavour: no fence, no separate flag. Every rank owns a mailbox
// [2 parities][nranks][NE_MAX entries][2 words] in its own HBM. A double travels as two 64-bit words {payload half |
// 32-bit sequence tag}; aligned 64-bit stores are single-copy atomic, so a reader that sees the expected tag in both words
// has the whole value — one NVLink one-way trip instead of store + system fence + flag. CTA 0 of rank r stores its entries
// into slot (parity, r) of EVERY rank's mailbox (its own included); every CTA of every rank then spins on the nranks slots
// of the LOCAL mailbox and adds them in rank order, so every CTA of every rank forms the bit-identical sum with no
// broadcast, no NCCL call and no kernel boundary.
// Tag and parity follow `seq`, the number of exchanges executed since peer_attach — a device-resident counter that persists
// across launches (levels may end early, updates may stop early: a per-launch formula would reuse a parity). Two parities
// suffice because exchanges strictly alternate: a rank's CTA 0 writes exchange k + 2 only after it received every peer's
// k + 1, which a peer's CTA 0 sends after its own grid barrier k + 1 — and every CTA of that peer passes that barrier only
// after it finished pulling exchange k.
#define PEER_SLOT_WORDS (NE_MAX * 2)  // u64 words per (parity, rank) slot
#define PEER_MAX_RANKS 8
struct PeerArgs {
  unsigned long long *const *mbox;  // device array: mailbox base of every rank (own entry = local memory)
  unsigned int *seq;                // device word: exchanges executed so far (same on every rank)
  int rank, nranks;
};

__device__ __forceinline__ void peer_push(const double *info, const PeerArgs &p, unsigned int seq) {
  const int tid = threadIdx.x;
  const unsigned int tag = seq + 1u;  // never 0 (the mailbox starts zeroed)
  const int par = seq & 1;
  if (tid < NE_MAX) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(info[tid]);
    const unsigned long long w0 = (bits << 32) | tag;                    // low half | tag
    const unsigned long long w1 = (bits & 0xffffffff00000000ull) | tag;  // high half | tag
    const size_t off = (size_t)(par * p.nranks + p.rank) * PEER_SLOT_WORDS + 2 * tid;
    for (int r = 0; r < p.nranks; r++) {
      unsigned long long *dst = p.mbox[r] + off;
      asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(w0) : "memory");
      asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(dst + 1), "l"(w1) : "memory");
    }
  }
}
__device__ __forceinline__ void peer_pull(double *info, const PeerArgs &p, unsigned int seq, WaitGuard &wg) {
  const int tid = threadIdx.x;
  const unsigned int tag = seq + 1u;
  const int par = seq & 1;
  if (tid < NE_MAX) {
    const unsigned long long *own = p.mbox[p.rank] + (size_t)par * p.nranks * PEER_SLOT_WORDS + 2 * tid;
    double s = 0.0;
    const unsigned long long t0 = globaltimer_ns();
    unsigned spins = 0;
    for (int r = 0; r < p.nranks; r++) {
      const unsigned long long *src = own + (size_t)r * PEER_SLOT_WORDS;
      unsigned long long a, b;
      for (;;) {
        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(a) : "l"(src) : "memory");
        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(b) : "l"(src + 1) : "memory");
        if (((unsigned int)a == tag && (unsigned int)b == tag) || wg.dead || wait_expired(wg, t0, spins)) break;
      }
      s += __longlong_as_double((long long)((b & 0xffffffff00000000ull) | (a >> 32)));
    }
    info[tid] = s;
  }
}

// Counting grid barrier over all CTAs of a cooperative launch: arrivals are release-increments, thread 0 of every CTA polls
// the same counter with acquire loads; the k-th barrier (k = 0, 1, ...) completes when it reaches (k + 1) * gridDim.x. The
// counter is zeroed for this launch by the previous launch (launches alternate between two counters). The waiting time does
// useful work: every thread but thread 0 runs `work` meanwhile. A variant with a separate release word written by the last
// arriver was measured and is ~1 us SLOWER per barrier (extra L2 hop), see profiles/README.md.
template <class F> __device__ __forceinline__ void grid_barrier_overlap(unsigned int *counter, unsigned int &epoch, WaitGuard &wg, F work) {
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int target = (epoch + 1) * gridDim.x;
    // release-increment: orders this CTA's earlier writes (made visible to thread 0 by the CTA barrier above) before the
    // arrival, without a separate membar; the acquire poll orders the other CTAs' writes before everything after it.
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    unsigned int v;
    const unsigned long long t0 = globaltimer_ns();
    unsigned spins = 0;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    } while (v < target && !wg.dead && !wait_expired(wg, t0, spins));
  } else {
    work();
  }
  epoch++;
  __syncthreads();
}

struct FusedSolveSmem {
  SolveSmem sm;
  SolveIO io;
  Ctrl ctrl;  // the CTA's working copy of the loop-control block
  WaitGuard wg;
};
static_assert(sizeof(FusedSolveSmem) % 8 == 0, "what follows it in shared memory holds doubles");

// Start of a persistent update, every CTA: loop control zeroed, waits armed, the literal-mode workspace (solve mode 1,
// parity checks) hooked up, the NEXT launch's barrier counter zeroed (no host memset per update) and the publisher's stats
// block cleared; then P, the current and the prior pose are staged, resident for the whole update.
__device__ __forceinline__ void persistent_prologue(FusedSolveSmem &fs, SolveLiteralScratch &lit, const SolveArgs &sa, Ctrl *ctrl, unsigned int *barrier_next,
                                                    void *stats, int stats_bytes) {
  if (threadIdx.x == 0) {
    Ctrl z;
    memset(&z, 0, sizeof(z));
    fs.ctrl = z;
    fs.wg.error_flag = &ctrl->comm_error, fs.wg.dead = false;
    fs.sm.W = lit.W, fs.sm.K = lit.K;
    if (blockIdx.x == 0) barrier_next[0] = 0u, barrier_next[32] = 0u;
  }
  if (!sa.no_publish && stats)
    for (int t = threadIdx.x; t < stats_bytes / 4; t += blockDim.x) reinterpret_cast<int *>(stats)[t] = 0;
  solve_load(fs.sm, fs.io, sa, false);
}

// The exchange of one iteration: this CTA's partial vector out (double-buffered by iteration parity, `part`), ONE grid
// barrier — warp 1 evaluates vec = state_propagat (-) state meanwhile (voxel_map.cpp:470, vio.cpp:1664) — then every CTA
// sums the partial columns in the same fixed order into fs.io.info and, with peer GPUs attached, adds the rank-ordered sum of
// every rank's vector. Phase stamp 3: all CTAs arrived.
template <int WARPS, int M, bool PEER>
__device__ __forceinline__ void exchange_info(FusedSolveSmem &fs, ReduceSmem<WARPS> &red, double D0, double D1, double cnt, double *part, int partial_stride,
                                              unsigned int *barrier, unsigned int &epoch, const PeerArgs &peer, unsigned int &seq,
                                              unsigned long long *stamps, int &sk) {
  store_partials<WARPS, M>(red, D0, D1, cnt, part, partial_stride);
  grid_barrier_overlap(barrier, epoch, fs.wg, [&]() {
    if ((threadIdx.x >> 5) == 1) boxminus_warp(fs.io.pr, fs.io.st, fs.sm.vec, threadIdx.x & 31);
  });
  stamp(stamps, sk);
  sum_partials<M>(part, partial_stride, gridDim.x, fs.io.info, WARPS);
  if (PEER) {
    __syncthreads();
    if (blockIdx.x == 0) peer_push(fs.io.info, peer, seq);
    peer_pull(fs.io.info, peer, seq, fs.wg);
    seq++;
  }
  __syncthreads();
}

// End of a persistent update, publisher thread 0: the loop control goes out with a sticky comm_error (a wait of any CTA may
// have expired), and the peer sequence is stored for the next launch.
template <bool PEER> __device__ __forceinline__ void publish_ctrl(FusedSolveSmem &fs, Ctrl *ctrl, const PeerArgs &peer, unsigned int seq) {
  fs.ctrl.comm_error = fs.wg.dead ? 1 : 0;
  const int err = *reinterpret_cast<volatile int *>(&ctrl->comm_error);
  *ctrl = fs.ctrl;
  if (err) ctrl->comm_error = 1;
  if (PEER) *peer.seq = seq;
}

template <bool PEER>
__global__ void __launch_bounds__(LIO_THREADS, 1) lio_update_kernel(const LioKernelArgs a, const SolveArgs sa_in, unsigned int *barrier, unsigned int *barrier_next, unsigned long long *stamps,
                                                                     size_t partial_parity_stride, const PeerArgs peer) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  LioSmem &sm = *reinterpret_cast<LioSmem *>(smem_raw);
  static_assert(sizeof(FusedSolveSmem) <= sizeof(sm.fs_raw), "solve state must fit");
  static_assert(sizeof(SolveLiteralScratch) <= sizeof(sm.rec), "literal scratch must fit in the record slots");
  FusedSolveSmem &fs = *reinterpret_cast<FusedSolveSmem *>(sm.fs_raw);
  SolveArgs sa = sa_in;
  const bool publisher = (blockIdx.x == gridDim.x - 1);
  sa.no_publish = !publisher;
  unsigned int epoch = 0;
  int lo, hi;
  lio_block_range(a.count, lo, hi);
  // the literal-mode workspace borrows the record slots and forces a re-stage
  persistent_prologue(fs, *reinterpret_cast<SolveLiteralScratch *>(&sm.rec[0][0][0]), sa, a.ctrl, barrier_next, sa.lio_stats, sizeof(esikf_lio_stats));
  lio_prior_consts(sm, a);
  unsigned int seq = PEER ? __ldcg(peer.seq) : 0u;
  lio_init_cold(sm, a);
  lio_init_barriers(sm);  // ends with a CTA barrier: fs.sm.P is in place
  if ((threadIdx.x >> 5) == LIO_WARPS - 1 && sa.solve_mode == 0) gain_setup<6>(fs.sm, 1.0, threadIdx.x & 31);  // loop invariants of the gain; first used after two CTA barriers
  lio_cov_consts(sm, fs.sm.P);  // state_.cov is only written after the loop (:489)
  int sk = 0;
  LaneCache lc;
  lane_cache_init(lc);
  for (int it = 0; it < sa.max_iterations; it++) {
    stamp(stamps, sk);  // 0: iteration start
    lio_pose_consts(sm, fs.io.st);
    __syncthreads();
    stamp(stamps, sk);  // 1: constants in place
    double D0 = 0.0, D1 = 0.0;
    int cnt = 0;
    // literal solve mode borrows the record slots as workspace: the per-point outputs cannot wait there for the last iteration
    lio_process_range(a, sm, lo, hi, D0, D1, cnt, lc, it == 0, sa.solve_mode == 1);
    if (stamps && it == 3) {  // measurement only: when did every CTA finish its slice of iteration 3?
      __syncthreads();
      if (threadIdx.x == 0) stamps[640 + blockIdx.x] = globaltimer_ns();
    }
    stamp(stamps, sk);  // 2: this CTA's warps issued their slice (CTA 0 / thread 0)
    exchange_info<LIO_WARPS, 6, PEER>(fs, sm.red, D0, D1, (double)cnt, a.partials + (size_t)(it & 1) * partial_parity_stride, a.partial_stride, barrier, epoch,
                                      peer, seq, stamps, sk);  // 3: all CTAs arrived
    stamp(stamps, sk);  // 4: information vector complete
    sa.dbg = (stamps && blockIdx.x == 0) ? stamps + sk + 1 : nullptr;  // 6: gain rows done, 7: boxplus done
    lio_solve_block(sa, fs.sm, fs.io, fs.ctrl);
    if (sa.solve_mode == 1) lane_cache_reset(lc);  // the literal workspace borrowed the record slots
    stamp(stamps, sk);  // 5: solved (state, loop control current in every CTA)
    sk += 2;            // 6, 7: spare
    if (fs.ctrl.stop) break;  // EKF_stop_flg (voxel_map.cpp:499)
  }
  if (sa.solve_mode != 1) lio_write_outputs(a, sm, lo, hi, lc);
  if (publisher && threadIdx.x == 0) publish_ctrl<PEER>(fs, a.ctrl, peer, seq);
}

// INVERSE: the inverse-compositional variant (vio/inverse_composition_en, src/vio.cpp:792-795, 1327-1518) in the same loop:
// every warp precomputes H_sub_inv of ITS patches when a level starts (precomputeReferencePatches; written and later read by
// the same lanes, so no barrier is involved) and the per-iteration build is vio_inverse_process_range.
template <bool PEER, bool INVERSE>
__global__ void __launch_bounds__(VIO_THREADS, 1) vio_update_kernel(const VioKernelArgs a, SolveArgs sa, unsigned int *barrier, unsigned int *barrier_next, unsigned long long *stamps,
                                                                     size_t partial_parity_stride, const PeerArgs peer, const VioInvArgs inv,
                                                                     const __grid_constant__ VioTma tma) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  VioSmem &sm = *reinterpret_cast<VioSmem *>(smem_raw);
  FusedSolveSmem &fs = *reinterpret_cast<FusedSolveSmem *>(smem_raw + sizeof(VioSmem));
  static_assert(sizeof(SolveLiteralScratch) <= sizeof(sm.rows), "literal scratch must fit in the row staging area");
  const bool publisher = (blockIdx.x == gridDim.x - 1);
  sa.no_publish = !publisher;
  unsigned int epoch = 0;
  int lo, hi;
  vio_block_range(a.count, lo, hi);
  const bool cached = (hi - lo) <= VIO_WARPS * VIO_KMAX;
  persistent_prologue(fs, *reinterpret_cast<SolveLiteralScratch *>(&sm.rows[0][0][0]), sa, a.ctrl, barrier_next, sa.vio_stats, sizeof(esikf_vio_stats));
  vio_cache_reset(sm);
  unsigned int seq = PEER ? __ldcg(peer.seq) : 0u;
  unsigned tma_phase = 0;  // parity of this warp's TMA barrier
  if (threadIdx.x < VIO_WARPS) mbar_init(&sm.tma_bar[threadIdx.x], 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  if ((threadIdx.x >> 5) == VIO_WARPS - 1 && sa.solve_mode == 0) gain_setup<7>(fs.sm, 1.0 / sa.img_point_cov, threadIdx.x & 31);  // loop invariants of the gain
  int slot = 0;
  for (int level = a.levels - 1; level >= 0; level--) {      // vio.cpp:790
    for (int it = 0; it < sa.max_iterations; it++) {          // :1536
      const int cur = slot++;  // counts executed iterations (a level may end early): the partial-buffer parity follows it
      int sk = 8 * ((a.levels - 1 - level) * sa.max_iterations + it);
      stamp(stamps, sk);
      vio_pose_consts(sm, a, fs.io.st);
      stamp(stamps, sk);
      double D0 = 0.0, D1 = 0.0, n_meas = 0.0;
      if (INVERSE) {
        if (it == 0)
          for (int lp = lo + (int)(threadIdx.x >> 5); lp < hi; lp += VIO_WARPS) vio_inverse_precompute_patch(a, inv, level, lp, threadIdx.x & 31);
        vio_inverse_process_range(a, inv, sm, level, lo, hi, fs.io.st, D0, D1, n_meas);
      } else {
        vio_process_range(a, sm, level, lo, hi, D0, D1, n_meas, cached, tma.enabled ? &tma : nullptr, &tma_phase);
      }
      stamp(stamps, sk);
      exchange_info<VIO_WARPS, 7, PEER>(fs, sm.red, D0, D1, n_meas, a.partials + (size_t)(cur & 1) * partial_parity_stride, a.partial_stride, barrier, epoch,
                                        peer, seq, stamps, sk);
      stamp(stamps, sk);
      sa.level = level, sa.slot_iter = it, sa.last_slot = 0;
      sa.dbg = (stamps && blockIdx.x == 0) ? stamps + sk + 1 : nullptr;  // 6: gain rows done, 7: boxplus done
      vio_solve_block(sa, fs.sm, fs.io, fs.ctrl);
      if (sa.solve_mode == 1) {  // the literal workspace borrowed the row area; nothing cached lives there
        __syncthreads();
      }
      stamp(stamps, sk);
      if (fs.ctrl.level_done) break;  // EKF_end (:1685)
    }
  }
  // state->cov -= G * state->cov (vio.cpp:800): a last-slot pass of the solve routine with the level already finished
  if (publisher) {
    __syncthreads();
    sa.level = 0, sa.slot_iter = 1, sa.last_slot = 1, sa.dbg = nullptr;
    if (threadIdx.x == 0) fs.ctrl.level_done = 1;
    __syncthreads();
    vio_solve_block(sa, fs.sm, fs.io, fs.ctrl);
    __syncthreads();
    if (threadIdx.x == 0) publish_ctrl<PEER>(fs, a.ctrl, peer, seq);
  }
}

}  // namespace esikf
