// sweepcore.cpp — TEST INFRASTRUCTURE: the parameter-sweep state machine (csrc/sim_core.cuh, SW = true) compiled with g++,
// so that sweeps can be checked against the oracle in the CPU-only container, as hostcore.cpp does for plain handles.  It is
// never part of, linked into, or reachable from the product library (librabft_simulator_b200/csrc/liblbft_b200.so).
#include <string>
#include <vector>

#include "../../librabft_simulator_b200/csrc/host_setup.hpp"
#include "../../librabft_simulator_b200/csrc/sim_core.cuh"

using namespace lbft;
static thread_local std::string g_err;

// Every instance reads its own set, as lbft_sweep_kernel does (32-instance tiles; the shared-memory queue is a per-call
// stand-in, like shared memory is per launch).
template <int NMAX, int QMODE>
static void run_all_sweep(const Params& P, std::vector<uint32_t>& state) {
  for (uint32_t inst = 0; inst < P.num_instances; inst++) {
    uint32_t tile = inst / 32, lane = inst % 32;
    TileMem<32> mem{state.data() + (size_t)tile * P.L.total_words * 32, lane};
    std::vector<uint32_t> sk(QMODE == 2 ? (size_t)P.L.queue_cap * 32 : 1);
    std::vector<uint16_t> sd(QMODE == 2 ? (size_t)P.L.queue_cap * 32 : 1);
    Core<TileMem<32>, NMAX, QMODE, FX_NONE, false, false, 1, false, false, false, true> core(P, mem, P.zig_x, P.zig_f, nullptr,
                                                                                          sk.data() + lane, sd.data() + lane);
    core.select_set(P.set_of[inst]);
    core.init(P.seeds[inst]);
    core.run();
    core.finalize(inst);
  }
}

extern "C" {
const char* sweepcore_last_error(void) { return g_err.c_str(); }

// Same contract as the product's lbft_create_sweep + lbft_run (include/lbft.h), with the outputs of its getters;
// layout_out (optional) receives [0] words per instance, [1] queue mode, [2] queue_cap, [3] payload_cap of the layout the
// sweep's instances share.
int sweepcore_run(const lbft_config* c, const lbft_param_set* sets, uint32_t num_sets, const uint32_t* set_of,
                  uint32_t* commit_counts, uint64_t* last_states, uint32_t* lc_round, uint32_t* counters, uint32_t* status,
                  uint32_t* layout_out) {
  HostSetup hs;
  if (!hs.build_sweep(*c, sets, num_sets, set_of)) { g_err = hs.error; return LBFT_ERR_INVALID; }
  Params P = hs.params;
  P.seeds = c->seeds;
  P.zig_x = hs.zig_x.data();
  P.zig_f = hs.zig_f.data();
  P.leader = hs.leader.data();
  P.weights = hs.weights.data();
  P.sweep_sets = hs.sets.data();
  P.set_of = hs.set_of.data();
  P.sweep_thr = hs.sweep_thr.data();
  P.sweep_duration = hs.sweep_duration.data();
  P.sweep_period = hs.sweep_period.data();
  P.num_sets = num_sets;
  std::vector<uint32_t> state((size_t)((c->num_instances + 31) / 32) * P.L.total_words * 32, 0xdeadbeefu);
  P.state = state.data();
  P.out_commit_counts = commit_counts;
  P.out_last_state = last_states;
  P.out_lc_round = lc_round;
  P.out_counters = counters;
  P.out_status = status;
  if (layout_out) {
    layout_out[0] = P.L.total_words;
    layout_out[1] = P.L.queue_scan;
    layout_out[2] = P.L.queue_cap;
    layout_out[3] = P.L.payload_cap;
  }
  const uint32_t N = c->num_nodes, q = P.L.queue_scan;
  if (q == 2) run_all_sweep<16, 2>(P, state);
  else if (q == 1) run_all_sweep<16, 1>(P, state);
  else if (q == 3) N <= 16 ? run_all_sweep<16, 3>(P, state) : (N <= 32 ? run_all_sweep<32, 3>(P, state) : run_all_sweep<64, 3>(P, state));
  else N <= 16 ? run_all_sweep<16, 0>(P, state) : (N <= 32 ? run_all_sweep<32, 0>(P, state) : run_all_sweep<64, 0>(P, state));
  return LBFT_OK;
}
}  // extern "C"
