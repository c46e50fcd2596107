// kernels.cuh — the two kernel templates over sim_core.cuh and the per-translation-unit launchers.
//
//   lbft_event_loop_kernel<NMAX, QMODE, FIXED, REC, RES>   one THREAD per instance, 32 instances per warp tile (large batches)
//   lbft_wide_kernel<NMAX, QMODE>                          one WARP per instance (small batches, large committees)
//
// Both do init -> event loop -> read-out in a single launch.  The instantiations are spread over several .cu files
// (k_fixed.cu, k_scan.cu, k_calendar.cu, k_heap.cu, k_wide.cu) so that they compile in parallel and the bench kernel
// can be rebuilt alone; lbft_api.cu only sees the launch_* functions declared at the end.  The kernels of parameter
// sweeps (Core SW = true) are defined in k_sweep.cu / k_sweep_wide.cu.
#pragma once
#include <cuda_runtime.h>

#include "sim_core.cuh"

namespace lbft {

#ifndef LBFT_NO_KS
#define LBFT_NO_KS 0  // A/B switch: 1 keeps the calendar's occupancy words in the instance's HBM block everywhere
#endif
// The wide kernels keep them in HBM: measured (profiles/r2n_ab_ks.txt) 8 192 x 64 on 8 lanes per instance 879 ms with the words in
// shared memory against 858 ms without (1 024 x 64 on a warp per instance: 313 vs 317 ms) — the words are L1-resident there
// anyway; the sparse-tile thread kernel gains 7.7 % (16 384 x 7: 42.4 vs 45.9 ms).
#ifndef LBFT_WIDE_KS
#define LBFT_WIDE_KS 0
#endif
LBFT_LAYOUT_FN uint32_t calendar_kmask_words(const Layout& L) { return (L.cal_times + 7) / 8; }
constexpr uint32_t kThrSmem = 256;  // doubles: delay thresholds held in shared memory when they fit

// Launch shapes of the thread-per-instance kernel.  QMODE 0/1/3: one-warp blocks, 14 resident per SM (2 048 tiles of a
// 65 536-instance batch over 148 SMs; <= 144 registers/thread keeps every tile resident).  QMODE 2: two-warp blocks, 7 per
// SM, so that the ziggurat/threshold tables (6 KB) are shared by two tiles and the per-tile event queues (queue_cap x 32 x
// 6 B) fit in the 227 KB of shared memory.
#ifndef LBFT_Q2_WARPS
#define LBFT_Q2_WARPS 2   // warps per block of the shared-memory-queue kernels (they share the 6 KB of tables)
#define LBFT_Q2_BLOCKS 7  // ... and blocks per SM: WARPS x BLOCKS = 14 tiles per SM, all 2 048 tiles of the bench batch resident
#endif
template <int QMODE>
struct LaunchShape {
  static constexpr int kThreads = QMODE == 2 ? 32 * LBFT_Q2_WARPS : 32;
  static constexpr int kBlocksPerSm = QMODE == 2 ? LBFT_Q2_BLOCKS : 14;
};

// TILE: instances per warp tile.  32 fills every lane; 8 / 4 ("sparse" tiles: the other lanes of the warp retire at once) trade
// lanes for warps when the batch is too small to fill the GPU with full warps — the instances of a warp serialise through
// each other's code paths, so a warp of 8 instances finishes far sooner than a warp of 32, and four times as many warps hide
// each other's latency.  Plain kernels over the calendar queue and the shared-memory queue (whose columns keep their
// 32-entry pitch); the state layout interleaves TILE instances.
template <int NMAX, int QMODE, int FX = FX_NONE, bool REC = false, bool RES = false, bool EP = false, bool TDS = false, int TILE = 32>
__global__ void __launch_bounds__(LaunchShape<QMODE>::kThreads, LaunchShape<QMODE>::kBlocksPerSm) lbft_event_loop_kernel(const __grid_constant__ Params P) {
  static_assert(TILE == 32 || ((QMODE == 3 || QMODE == 2) && !REC && !RES && !EP && !TDS), "sparse tiles: plain kernels over the calendar / shared-memory queue");
  // The ziggurat layers are indexed by a random byte per lane: a per-block shared-memory copy (4 KB) serves the 32
  // scattered 8-byte reads of a warp in ~1-2 wavefronts; reading them through L1 from global memory instead was
  // measured 1.5x slower for the whole kernel (44.1 vs 28.9 ms).
  __shared__ double s_zx[257];
  __shared__ double s_zf[257];
  __shared__ double s_thr[kThrSmem];  // delay thresholds (same scattered access pattern), when they fit
  extern __shared__ uint32_t s_queue[];  // QMODE 2: per warp [queue_cap][32] u32 keys, then [queue_cap][32] u16 payload words
                                         // QMODE 3, sparse tiles: per warp [kmask words][TILE] calendar occupancy words
  for (int i = threadIdx.x; i < 257; i += blockDim.x) {
    s_zx[i] = P.zig_x[i];
    s_zf[i] = P.zig_f[i];
  }
  const bool thr_fits = P.delay_kmax != 0 && P.delay_kmax + 2 <= kThrSmem;
  if (thr_fits)
    for (uint32_t i = threadIdx.x; i < P.delay_kmax + 2; i += blockDim.x) s_thr[i] = P.delay_thr[i];
  __syncthreads();
  const uint32_t gthread = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t tile = gthread >> 5, lane = gthread & 31;
  const uint32_t inst = tile * TILE + lane;
  if (lane >= TILE || inst >= P.num_instances) return;
  const uint32_t total_words = FX ? fixed_layout(FX).total_words : P.L.total_words;
  TileMem<TILE> mem{P.state + (size_t)tile * total_words * TILE, lane};
  uint32_t* sk = nullptr;
  uint16_t* sd = nullptr;
  if (QMODE == 2) {
    const uint32_t warp = threadIdx.x >> 5, qcap = P.L.queue_cap;
    uint32_t* base = s_queue + (size_t)warp * (qcap * 32 + qcap * 16);  // keys (qcap*32 words) + payload (qcap*32 halves)
    sk = base + lane;
    sd = reinterpret_cast<uint16_t*>(base + qcap * 32) + lane;
  }
  // sparse tiles over the calendar queue: the kind-occupancy words of the tile's instances in shared memory, a column per
  // lane (sim_core.cuh KS; the host only selects sparse tiles when 14 warps' worth fits, host_setup.hpp)
  constexpr bool KS = QMODE == 3 && TILE < 32 && !LBFT_NO_KS;
  Core<TileMem<TILE>, NMAX, QMODE, FX, REC, RES, 1, EP, TDS, KS> core(P, mem, s_zx, s_zf, thr_fits ? s_thr : P.delay_thr, sk, sd);
  if (KS) core.km = s_queue + (size_t)(threadIdx.x >> 5) * calendar_kmask_words(FX ? fixed_layout(FX) : P.L) * TILE + lane;
  if (RES && (P.run_flags & 1u)) core.restore_regs();  // a later lbft_run_until: continue where the last launch stopped
  else core.init(P.seeds[inst]);
  core.run();
  core.finalize(inst);
  if (RES) core.save_regs();
}

// ---- a group of G lanes per instance ("wide") ---------------------------------------------------------------------
// wide_warps(G) warps per block, 32 / G instances per warp (instance = global group index; the hardware block scheduler hands
// out the next block as soon as one retires, which is the work queue SURVEY §8e asks for).  The state of an instance is one
// contiguous extent (TileMem<1>: stride 1), tables are read through L1 (every lane of a group reads the same element), the
// shared-memory queue of QMODE 2 and the fan-out scratch are per group.
// Warps per block: four when a warp carries several instances; ONE when a warp is an instance (G = 32): a block is then a
// single instance, its index arithmetic folds away (5 192 instead of 5 600 SASS instructions) and blocks retire one by one —
// measured (profiles/r2p_ab_wide_warps.txt) 1 024 x 4: 2.48 ms against 3.81 with four-warp blocks, a lone instance 3.66 against
// 4.44 ms; 8 lanes per instance (8 192 x 64) is indifferent: 838 / 842 / 840 ms for 4 / 2 / 1 warps.
#ifndef LBFT_WIDE_WARPS
#define LBFT_WIDE_WARPS 4  // (blocks of the G < 32 kernels)
#endif
LBFT_LAYOUT_FN int wide_warps(int g) { return g == 32 ? 1 : LBFT_WIDE_WARPS; }
// blocks per SM the register allocation is bounded for: 16 warps per SM, <= 128 registers
LBFT_LAYOUT_FN int wide_blocks_per_sm(int g) { return 16 / wide_warps(g); }

// Shared memory of one group: [scratch][QMODE 2: queue keys, queue payload halves][SMEM: the instance state]
LBFT_LAYOUT_FN uint32_t wide_scratch_words() { return (uint32_t)((sizeof(WideScratch) + 7) / 8 * 2); }
LBFT_LAYOUT_FN uint32_t wide_queue_words(uint32_t queue_cap, int qmode) {
  return qmode == 2 ? ((queue_cap + (queue_cap + 1) / 2 + 1) & ~1u) : 0u;  // even: what follows holds 64-bit entries
}
LBFT_LAYOUT_FN uint32_t wide_smem_words_per_group(const Layout& L, int qmode, bool smem_state) {
  return wide_scratch_words() + wide_queue_words(L.queue_cap, qmode) + (smem_state ? ((L.total_words + 1) & ~1u) : 0u) +
         (qmode == 3 && LBFT_WIDE_KS ? ((calendar_kmask_words(L) + 1) & ~1u) : 0u);  // QMODE 3: the calendar's occupancy words (sim_core.cuh KS)
}

// SMEM: the instance's state words live in shared memory for the whole run; only the chain table (and the epoch table) is
// copied to the instance's global extent at the end, for lbft_commit_log / lbft_commit_logs.
template <int NMAX, int QMODE, bool SMEM, int G, bool EP = false, int FX = FX_NONE>
__global__ void __launch_bounds__(wide_warps(G) * 32, wide_blocks_per_sm(G)) lbft_wide_kernel(const __grid_constant__ Params P) {
  extern __shared__ __align__(8) uint32_t s_wide[];
  constexpr uint32_t kPerBlock = wide_warps(G) * 32 / G;
  const uint32_t grp = threadIdx.x / G, wl = threadIdx.x % G;
  const uint32_t inst = blockIdx.x * kPerBlock + grp;
  if (inst >= P.num_instances) return;  // whole groups leave together: everything below is group-uniform
  const Layout KL = FX ? fixed_layout(FX) : P.L;
  uint32_t* base = s_wide + (size_t)grp * wide_smem_words_per_group(KL, QMODE, SMEM);
  WideScratch* ws = reinterpret_cast<WideScratch*>(base);
  uint32_t* sk = base + wide_scratch_words();
  uint16_t* sd = reinterpret_cast<uint16_t*>(sk + KL.queue_cap);
  uint32_t* gstate = P.state + (size_t)inst * KL.total_words;
  uint32_t* state = SMEM ? sk + wide_queue_words(KL.queue_cap, QMODE) : gstate;
  TileMem<1> mem{state, 0};
  constexpr bool KS = QMODE == 3 && LBFT_WIDE_KS;
  Core<TileMem<1>, NMAX, QMODE, FX, false, false, G, EP, false, KS> core(P, mem, P.zig_x, P.zig_f, P.delay_thr, sk, sd);
  if (KS) core.km = base + wide_scratch_words();  // (QMODE 3 has no shared-memory queue and no shared-memory state: the words follow the scratch)
  core.wl = wl;
  core.gm = G == 32 ? 0xffffffffu : (((1u << (G & 31)) - 1u) << ((threadIdx.x & 31u) & ~(uint32_t)(G - 1)));
  core.ws = ws;
  core.init(P.seeds[inst]);
  core.run();
  core.finalize(inst);
  if (SMEM) {
    __syncwarp(core.gm);
    for (uint32_t w = P.L.chain_base + wl; w < P.L.chain_base + 2 * P.L.round_cap; w += G) gstate[w] = state[w];
    if (EP)
      for (uint32_t w = wl; w < P.L.epochs; w += G) gstate[P.L.einit_base + w] = state[P.L.einit_base + w];
  }
}

// What the host decided to launch for a handle (host_setup.hpp / lbft_api.cu select_kernel).
struct KernelSel {
  bool wide;   // lbft_wide_kernel instead of lbft_event_loop_kernel
  bool smem;   // wide kernel: instance state in shared memory
  int group;   // wide kernel: lanes per instance (8 / 32)
  bool epochs; // Layout::epochs > 1: the instantiation with the epoch machinery (plain kernels only)
  bool tds;    // LBFT_FLAG_TRUE_DATA_SYNC (plain single-epoch thread kernels only)
  int tile;    // thread kernel: instances per warp tile (32; 8 / 4 = sparse tiles, plain calendar-queue kernels)
  int nmax;    // 16 / 32 / 64: width of the author masks
  int qmode;   // Layout::queue_scan
  int fixed;   // FX_* (sim_params.h): the instantiation with that compile-time layout; FX_NONE = generic
  bool rec, res;
  bool sweep;  // parameter sweep (lbft_create_sweep): lbft_sweep_kernel / lbft_sweep_wide_kernel (k_sweep*.cu)
};

// One per translation unit; each returns cudaErrorInvalidValue if the selection is not one of its instantiations.
cudaError_t launch_fixed(const KernelSel& k, const Params& P, cudaStream_t stream);
cudaError_t launch_scan(const KernelSel& k, const Params& P, cudaStream_t stream);
cudaError_t launch_calendar(const KernelSel& k, const Params& P, cudaStream_t stream);
cudaError_t launch_heap(const KernelSel& k, const Params& P, cudaStream_t stream);
cudaError_t launch_wide(const KernelSel& k, const Params& P, cudaStream_t stream);
cudaError_t launch_sweep(const KernelSel& k, const Params& P, cudaStream_t stream);
cudaError_t launch_sweep_wide(const KernelSel& k, const Params& P, cudaStream_t stream);

// Shared by the launchers of the thread-per-instance kernel.
template <int NMAX, int QM, int TILE, int FX = FX_NONE>
inline cudaError_t launch_sparse_tiles(const Params& P, cudaStream_t stream) {
  constexpr int T = LaunchShape<QM>::kThreads;
  const uint32_t tiles = (P.num_instances + TILE - 1) / TILE, blocks = (tiles * 32 + T - 1) / T;
  const size_t dyn = QM == 2 ? (size_t)(T / 32) * P.L.queue_cap * (32 * 4 + 32 * 2)
                             : (size_t)(T / 32) * calendar_kmask_words(P.L) * TILE * sizeof(uint32_t);  // (QMODE 3: sim_core.cuh KS)
  if (dyn > 48 * 1024) return cudaErrorInvalidValue;  // (the host keeps sparse tiles to horizons whose occupancy words fit)
  lbft_event_loop_kernel<NMAX, QM, FX, false, false, false, false, TILE><<<blocks, T, dyn, stream>>>(P);
  return cudaGetLastError();
}
template <int NMAX, int QM>
inline cudaError_t launch_thread_variants(const KernelSel& k, const Params& P, cudaStream_t stream) {
  constexpr int T = LaunchShape<QM>::kThreads;
  const uint32_t blocks = (P.num_instances + T - 1) / T;
  const size_t dyn = QM == 2 ? (size_t)(T / 32) * P.L.queue_cap * (32 * 4 + 32 * 2) : 0;
  if (k.tds) {
    if (k.rec || k.res || k.epochs) return cudaErrorInvalidValue;  // (refused at lbft_create)
    lbft_event_loop_kernel<NMAX, QM, FX_NONE, false, false, false, true><<<blocks, T, dyn, stream>>>(P);
  } else if (k.epochs) {
    if (k.rec || k.res) return cudaErrorInvalidValue;  // (refused at lbft_create)
    lbft_event_loop_kernel<NMAX, QM, FX_NONE, false, false, true><<<blocks, T, dyn, stream>>>(P);
  } else if (k.rec && k.res) lbft_event_loop_kernel<NMAX, QM, FX_NONE, true, true><<<blocks, T, dyn, stream>>>(P);
  else if (k.res) lbft_event_loop_kernel<NMAX, QM, FX_NONE, false, true><<<blocks, T, dyn, stream>>>(P);
  else if (k.rec) lbft_event_loop_kernel<NMAX, QM, FX_NONE, true><<<blocks, T, dyn, stream>>>(P);
  else lbft_event_loop_kernel<NMAX, QM><<<blocks, T, dyn, stream>>>(P);
  return cudaGetLastError();
}

template <int NMAX, int QM, bool SMEM, int G, bool EP, int FX = FX_NONE>
inline cudaError_t launch_wide_variant(const Params& P, cudaStream_t stream) {
  constexpr uint32_t kPerBlock = wide_warps(G) * 32 / G;
  const uint32_t blocks = (P.num_instances + kPerBlock - 1) / kPerBlock;
  const size_t dyn = (size_t)kPerBlock * wide_smem_words_per_group(P.L, QM, SMEM) * sizeof(uint32_t);
  static size_t attr_set = 48 * 1024;  // (per instantiation; two threads racing set the same or a larger value)
  if (dyn > attr_set) {
    cudaError_t e = cudaFuncSetAttribute(lbft_wide_kernel<NMAX, QM, SMEM, G, EP, FX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return e;
    attr_set = dyn;
  }
  lbft_wide_kernel<NMAX, QM, SMEM, G, EP, FX><<<blocks, wide_warps(G) * 32, dyn, stream>>>(P);
  return cudaGetLastError();
}
// the lanes-per-instance / epoch dimensions of an instantiation family (the host only selects these combinations)
template <int NMAX, int QM, bool SMEM>
inline cudaError_t launch_wide_groups(const KernelSel& k, const Params& P, cudaStream_t stream) {
  if (k.epochs) {
    if (SMEM || k.group != 32) return cudaErrorInvalidValue;
    return launch_wide_variant<NMAX, QM, false, 32, true>(P, stream);
  }
  if (k.fixed == FX_COMMITTEE64) {  // (lbft_api.cu select_kernel: 64 authors, calendar queue, 8 lanes per instance, state in HBM)
    if (NMAX != 64 || QM != 3 || SMEM || k.group != 8) return cudaErrorInvalidValue;
    return launch_wide_variant<64, 3, false, 8, false, (NMAX == 64 && QM == 3 && !SMEM) ? FX_COMMITTEE64 : FX_NONE>(P, stream);
  }
  if (k.group == 8) return launch_wide_variant<NMAX, QM, SMEM, 8, false>(P, stream);
  return launch_wide_variant<NMAX, QM, SMEM, 32, false>(P, stream);
}

}  // namespace lbft
