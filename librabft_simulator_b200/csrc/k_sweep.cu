// k_sweep.cu — thread-per-instance kernels of parameter sweeps (lbft_create_sweep; sim_core.cuh SW): 32 instances per warp
// tile, each with its own parameter set.  Generic layouts only (no FX), plain one-shot runs.
#include "kernels.cuh"
namespace lbft {

// lbft_event_loop_kernel's plain full-tile path, except that the delay thresholds stay in global memory: the instances of a
// block belong to different sets, so one shared-memory copy of a table cannot serve them.  They are read through L1.
template <int NMAX, int QMODE>
__global__ void __launch_bounds__(LaunchShape<QMODE>::kThreads, LaunchShape<QMODE>::kBlocksPerSm) lbft_sweep_kernel(const __grid_constant__ Params P) {
  __shared__ double s_zx[257];
  __shared__ double s_zf[257];
  extern __shared__ uint32_t s_queue[];  // QMODE 2: per warp [queue_cap][32] u32 keys, then [queue_cap][32] u16 payload words
  for (int i = threadIdx.x; i < 257; i += blockDim.x) {
    s_zx[i] = P.zig_x[i];
    s_zf[i] = P.zig_f[i];
  }
  __syncthreads();
  const uint32_t inst = blockIdx.x * blockDim.x + threadIdx.x;
  if (inst >= P.num_instances) return;
  const uint32_t tile = inst >> 5, lane = inst & 31;
  TileMem<32> mem{P.state + (size_t)tile * P.L.total_words * 32, lane};
  uint32_t* sk = nullptr;
  uint16_t* sd = nullptr;
  if (QMODE == 2) {
    const uint32_t warp = threadIdx.x >> 5, qcap = P.L.queue_cap;
    uint32_t* base = s_queue + (size_t)warp * (qcap * 32 + qcap * 16);
    sk = base + lane;
    sd = reinterpret_cast<uint16_t*>(base + qcap * 32) + lane;
  }
  Core<TileMem<32>, NMAX, QMODE, FX_NONE, false, false, 1, false, false, false, true> core(P, mem, s_zx, s_zf, nullptr, sk, sd);
  core.select_set(P.set_of[inst]);
  core.init(P.seeds[inst]);
  core.run();
  core.finalize(inst);
}

template <int NMAX, int QM>
static cudaError_t launch_sweep_thread(const Params& P, cudaStream_t stream) {
  constexpr int T = LaunchShape<QM>::kThreads;
  const uint32_t blocks = (P.num_instances + T - 1) / T;
  const size_t dyn = QM == 2 ? (size_t)(T / 32) * P.L.queue_cap * (32 * 4 + 32 * 2) : 0;
  lbft_sweep_kernel<NMAX, QM><<<blocks, T, dyn, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_sweep(const KernelSel& k, const Params& P, cudaStream_t stream) {
  if (!k.sweep || k.wide || k.tile != 32 || k.fixed || k.rec || k.res || k.epochs || k.tds) return cudaErrorInvalidValue;
  switch (k.qmode) {
    case 2: return launch_sweep_thread<16, 2>(P, stream);
    case 1: return launch_sweep_thread<16, 1>(P, stream);
    case 3:
      if (k.nmax == 16) return launch_sweep_thread<16, 3>(P, stream);
      if (k.nmax == 32) return launch_sweep_thread<32, 3>(P, stream);
      return launch_sweep_thread<64, 3>(P, stream);
    default:
      if (k.nmax == 16) return launch_sweep_thread<16, 0>(P, stream);
      if (k.nmax == 32) return launch_sweep_thread<32, 0>(P, stream);
      return launch_sweep_thread<64, 0>(P, stream);
  }
}

}  // namespace lbft
