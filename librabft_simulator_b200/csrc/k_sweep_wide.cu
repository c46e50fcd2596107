// k_sweep_wide.cu — lane-group-per-instance kernels of parameter sweeps (lbft_create_sweep; sim_core.cuh SW): small
// batches, large committees, and the shapes where a plain handle would take sparse thread-kernel tiles.
#include "kernels.cuh"
namespace lbft {

// lbft_wide_kernel without the epoch machinery and the compile-time layouts; each instance reads its own set.
template <int NMAX, int QMODE, bool SMEM, int G>
__global__ void __launch_bounds__(wide_warps(G) * 32, wide_blocks_per_sm(G)) lbft_sweep_wide_kernel(const __grid_constant__ Params P) {
  extern __shared__ __align__(8) uint32_t s_wide[];
  constexpr uint32_t kPerBlock = wide_warps(G) * 32 / G;
  const uint32_t grp = threadIdx.x / G, wl = threadIdx.x % G;
  const uint32_t inst = blockIdx.x * kPerBlock + grp;
  if (inst >= P.num_instances) return;  // whole groups leave together
  uint32_t* base = s_wide + (size_t)grp * wide_smem_words_per_group(P.L, QMODE, SMEM);
  WideScratch* ws = reinterpret_cast<WideScratch*>(base);
  uint32_t* sk = base + wide_scratch_words();
  uint16_t* sd = reinterpret_cast<uint16_t*>(sk + P.L.queue_cap);
  uint32_t* gstate = P.state + (size_t)inst * P.L.total_words;
  uint32_t* state = SMEM ? sk + wide_queue_words(P.L.queue_cap, QMODE) : gstate;
  TileMem<1> mem{state, 0};
  constexpr bool KS = QMODE == 3 && LBFT_WIDE_KS;
  Core<TileMem<1>, NMAX, QMODE, FX_NONE, false, false, G, false, false, KS, true> core(P, mem, P.zig_x, P.zig_f, nullptr, sk, sd);
  if (KS) core.km = base + wide_scratch_words();
  core.wl = wl;
  core.gm = G == 32 ? 0xffffffffu : (((1u << (G & 31)) - 1u) << ((threadIdx.x & 31u) & ~(uint32_t)(G - 1)));
  core.ws = ws;
  core.select_set(P.set_of[inst]);
  core.init(P.seeds[inst]);
  core.run();
  core.finalize(inst);
  if (SMEM) {
    __syncwarp(core.gm);
    for (uint32_t w = P.L.chain_base + wl; w < P.L.chain_base + 2 * P.L.round_cap; w += G) gstate[w] = state[w];
  }
}

template <int NMAX, int QM, bool SMEM, int G>
static cudaError_t launch_sweep_wide_variant(const Params& P, cudaStream_t stream) {
  constexpr uint32_t kPerBlock = wide_warps(G) * 32 / G;
  const uint32_t blocks = (P.num_instances + kPerBlock - 1) / kPerBlock;
  const size_t dyn = (size_t)kPerBlock * wide_smem_words_per_group(P.L, QM, SMEM) * sizeof(uint32_t);
  static size_t attr_set = 48 * 1024;  // (per instantiation; two threads racing set the same or a larger value)
  if (dyn > attr_set) {
    cudaError_t e = cudaFuncSetAttribute(lbft_sweep_wide_kernel<NMAX, QM, SMEM, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return e;
    attr_set = dyn;
  }
  lbft_sweep_wide_kernel<NMAX, QM, SMEM, G><<<blocks, wide_warps(G) * 32, dyn, stream>>>(P);
  return cudaGetLastError();
}
template <int NMAX, int QM, bool SMEM>
static cudaError_t launch_sweep_groups(const KernelSel& k, const Params& P, cudaStream_t stream) {
  return k.group == 8 ? launch_sweep_wide_variant<NMAX, QM, SMEM, 8>(P, stream) : launch_sweep_wide_variant<NMAX, QM, SMEM, 32>(P, stream);
}

cudaError_t launch_sweep_wide(const KernelSel& k, const Params& P, cudaStream_t stream) {
  if (!k.sweep || !k.wide || k.fixed || k.rec || k.res || k.epochs || k.tds) return cudaErrorInvalidValue;
  switch (k.qmode) {
    case 2: return k.smem ? launch_sweep_groups<16, 2, true>(k, P, stream) : launch_sweep_groups<16, 2, false>(k, P, stream);
    case 1: return launch_sweep_groups<16, 1, false>(k, P, stream);
    case 3:
      if (k.nmax == 16) return launch_sweep_groups<16, 3, false>(k, P, stream);
      if (k.nmax == 32) return launch_sweep_groups<32, 3, false>(k, P, stream);
      return launch_sweep_groups<64, 3, false>(k, P, stream);
    default:
      if (k.nmax == 16) return launch_sweep_groups<16, 0, false>(k, P, stream);
      if (k.nmax == 32) return launch_sweep_groups<32, 0, false>(k, P, stream);
      return launch_sweep_groups<64, 0, false>(k, P, stream);
  }
}

}  // namespace lbft
