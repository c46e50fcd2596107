// sim_params.h — launch-uniform parameters and the per-instance HBM layout of the batched
// LibraBFTv2 simulator.  Shared by the host runtime (lbft_api.cu) and the device core
// (sim_core.cuh).  Plain C++ (no CUDA types) so that the host test harness can include it too.
//
// HBM layout ("warp tiles"): instances are grouped 32 to a tile; a tile is `total_words` rows of
// 32 u32 lanes, i.e. word w of the instance in lane l of tile t lives at
//      state[(t * total_words + w) * 32 + l].
// Whenever the 32 lanes of a warp touch the same logical word, the access is one fully coalesced
// 128-byte line; a tile is one contiguous (total_words * 128)-byte extent that a single bulk copy
// can stage into shared memory.
#pragma once
#include <stdint.h>

namespace lbft {

enum : uint32_t { EV_NOTIFY = 0, EV_REQUEST = 1, EV_RESPONSE = 2, EV_TIMER = 3 };

// Per-node scalar fields, one u32 word each (node.rs:28-45, record_store.rs:93-119,
// pacemaker.rs:58-78, simulator.rs:53-59, simulated_context.rs:74-83 in round-id form).
enum NodeField : uint32_t {
  F_STARTUP = 0,   // SimulatedNode.startup_time (global ms)
  F_IGNORE,        // SimulatedNode.ignore_scheduled_updates_until
  F_CUR,           // record_store.current_round
  F_HQC,           // highest_quorum_certificate_round (QC identified by its round)
  F_HTC,           // highest_timeout_certificate_round
  F_HCR,           // highest_committed_round
  F_HCC,           // round of highest_commit_certificate (0 = None)
  F_LVR,           // node.latest_voted_round
  F_LOCKED,        // node.locked_round
  F_PMR,           // pacemaker.active_round
  F_PM_START,      // pacemaker.active_round_start_time (node-local ms)
  F_PM_DUR,        // pacemaker.active_round_duration
  F_PM_PERIOD,     // (lambda * duration) as i64
  F_LQA,           // node.latest_query_all_time
  F_TRK_HCR,       // tracker.highest_committed_round
  F_TRK_TIME,      // tracker.latest_commit_time
  F_FLAGS,         // bit0 current_proposed_block.is_some, bits1-2 election, bit3 has TC, bits8-15 active_leader (0xff None),
                   // bits16-20 node.epoch_id, bits21-25 pacemaker.active_epoch, bits26-30 tracker.epoch_id (all 0 unless the
                   // configuration can reach an epoch change, Layout::epochs > 1)
  F_NEXT_CMD,      // context.next_fetched_command_index
  F_LC_ROUND,      // block whose state is last_committed_ledger_state, as a GLOBAL round id epoch * rspan + round (0 = genesis)
  F_COMMITS,       // committed_history().len()
  F_BALLOT,        // weight of votes for the (single) block of the current round
  F_TOW,           // current_timeouts_weight
  F_TC_ROUND,      // round of highest_timeout_certificate
  F_LAST_TIMER,    // time of the most recently pushed UpdateTimerEvent (for exact de-duplication)
  F_NSCALAR
};
enum : uint32_t {
  FL_PROPOSED = 1u,
  FL_ELECTION_SHIFT = 1,  // 0 Ongoing, 1 Won, 2 Closed
  FL_ELECTION_MASK = 3u << 1,
  FL_HAS_TC = 1u << 3,
  FL_LEADER_SHIFT = 8,
  FL_LEADER_NONE = 0xffu,
  FL_EPOCH_SHIFT = 16,      // node.epoch_id (node.rs:32)
  FL_PM_EPOCH_SHIFT = 21,   // pacemaker.active_epoch (pacemaker.rs:60)
  FL_TRK_EPOCH_SHIFT = 26,  // tracker.epoch_id (node.rs:354)
  FL_EPOCH_BITS = 31u,
  MAX_EPOCHS = 32
};

struct Layout {
  uint32_t num_nodes;
  uint32_t mask_words;   // 1 (N<=32) or 2 (N<=64): author bitmasks
  uint32_t hcbr_words;   // ceil(N/2): per-author u16 highest_certified_block_round of a timeout
  uint32_t rset_words;   // round_cap/32: per-round bitsets
  uint32_t round_cap, queue_cap, payload_cap, part_windows;
  uint32_t queue_scan;   // QMODE: 0 binary heap (3-word entries) | 1 scan queue, 64-bit entries in HBM | 2 scan queue, 32+16-bit
                         // entries in shared memory | 3 calendar queue (per-(time, kind) FIFO lists) in HBM
  uint32_t cal_kmask, cal_ht, cal_times;  // QMODE 3: kind-occupancy nibbles (8 times per word), head|tail<<16 per (time, kind)
  // word offsets inside a node block
  uint32_t n_vmask, n_tmask, n_tcmask, n_thcbr, n_tchcbr, n_hasblk, n_hasqc, n_pend, node_words;
  // word offsets inside an instance
  uint32_t node_base, created_base /* per-round "block exists" / "QC exists" bitsets */, qcmade_base, chain_base,
      part_base, heap_time, heap_key, heap_data, pay_base, pay_words, total_words;
  // payload slot: [0] hcc | hqc<<16  [1] cur_round | tc_round<<16  [2] refcount | flags<<16 (bit0 vote, bit1 proposal)
  //               [3..] tc mask, cur mask, tc hcbr[], cur hcbr[]
  uint32_t p_tcmask, p_curmask, p_tchcbr, p_curhcbr;
  // Epochs (node.rs:329-348).  A record is identified by (epoch, round): its GLOBAL round id is epoch * rspan + round, and
  // the per-round tables (chain, the three bitsets of a node) cover round_cap = epochs * rspan global ids.  epochs == 1
  // (commands_per_epoch cannot be reached within the horizon — every BASELINE configuration): rspan == round_cap and
  // nothing changes.  einit_base: per-instance table [epochs] of the global id of the block whose state is the epoch's
  // initial state (0 for epoch 0).
  uint32_t rspan, epochs, einit_base;
  // LBFT_FLAG_TRUE_DATA_SYNC: payload slots carry a per-round bitset behind the notification fields — the requester's
  // known QC rounds in a request, the rounds whose block + QC the responder hands over in a response.
  uint32_t p_rounds, tds;
};

#if defined(__CUDACC__)
#define LBFT_LAYOUT_FN __host__ __device__ constexpr
#else
#define LBFT_LAYOUT_FN constexpr
#endif
// Save area of a resumable instance: [0, RES_REG_WORDS) the per-instance registers of Core (save_regs/restore_regs);
// then round_cap words of scratch for finalize() (the event queue is still live, so it cannot be borrowed as in a
// one-shot run); QMODE 2 only: queue_cap key words + (queue_cap + 1) / 2 words of packed 16-bit payloads — the
// shared-memory queue between two launches.
constexpr uint32_t RES_REG_WORDS = 40;

LBFT_LAYOUT_FN Layout make_layout(uint32_t N, uint32_t round_cap, uint32_t queue_cap, uint32_t payload_cap, uint32_t part_windows,
                          uint32_t queue_scan, uint32_t max_clock = 0, bool record_rs = false, bool resumable = false, uint32_t epochs = 1,
                          bool true_data_sync = false) {
  Layout L{};
  L.epochs = epochs;
  L.rspan = round_cap;       // rounds representable per epoch
  round_cap *= epochs;       // global round ids
  L.queue_scan = queue_scan;
  L.num_nodes = N;
  L.mask_words = N > 32 ? 2 : 1;
  L.hcbr_words = (N + 1) / 2;
  L.round_cap = round_cap;
  L.rset_words = round_cap / 32;
  L.queue_cap = queue_cap;
  L.payload_cap = payload_cap;
  L.part_windows = part_windows;
  uint32_t w = F_NSCALAR;
  L.n_vmask = w; w += L.mask_words;
  L.n_tmask = w; w += L.mask_words;
  L.n_tcmask = w; w += L.mask_words;
  L.n_thcbr = w; w += L.hcbr_words;
  L.n_tchcbr = w; w += L.hcbr_words;
  L.n_hasblk = w; w += L.rset_words;
  L.n_hasqc = w; w += L.rset_words;
  L.n_pend = w; w += L.rset_words;
  L.node_words = w;
  uint32_t o = 0;
  L.node_base = o; o += N * L.node_words;
  L.created_base = o; o += L.rset_words;
  L.qcmade_base = o; o += L.rset_words;
  L.chain_base = o; o += 2 * round_cap;  // [2r] prev | cmd<<16, [2r+1] time
  L.part_base = o; o += 4 * part_windows;  // t0, t1, mask lo, mask hi
  o = (o + 1) & ~1u;  // 64-bit entries of the scan queue need an even word offset
  L.heap_time = o; o += queue_cap;
  L.heap_key = o; o += queue_cap;
  if (queue_scan == 0) { L.heap_data = o; o += queue_cap; }
  if (queue_scan == 3) {  // heap_time = pool `next` links, heap_key = pool payload words
    L.cal_times = max_clock + 1;
    L.cal_kmask = o; o += (L.cal_times + 7) / 8;
    L.cal_ht = o; o += L.cal_times * 4;
  }
  L.p_tcmask = 3;
  L.p_curmask = L.p_tcmask + L.mask_words;
  L.p_tchcbr = L.p_curmask + L.mask_words;
  L.p_curhcbr = L.p_tchcbr + L.hcbr_words;
  L.pay_words = L.p_curhcbr + L.hcbr_words;
  L.p_rounds = L.pay_words;
  L.tds = true_data_sync ? 1u : 0u;
  if (true_data_sync) L.pay_words += L.rset_words;
  L.pay_base = o; o += payload_cap * L.pay_words;
  // DataWriter round-switch table (data_writer.rs:14), only when recording (LBFT_FLAG_ROUND_SWITCHES): [node][round 0..round_cap]
  // = pop time + 1 (pops are at t >= 1; 0 = never seen), num_nodes * (round_cap + 1) words at the END of the instance, found
  // with rs_table_base() — deliberately not a Layout field, so that Layout / Params keep the exact shape the
  // compile-time-layout kernel was tuned with.
  if (record_rs) o += N * (round_cap + 1);
  // Resumable runs (LBFT_FLAG_RESUMABLE): a per-instance save area after that table, see res_area_words() below.
  if (resumable) o += RES_REG_WORDS + round_cap + (queue_scan == 2 ? queue_cap + (queue_cap + 1) / 2 : 0);
  // (appended last so that single-epoch layouts keep every other offset)
  L.einit_base = o;
  if (epochs > 1) o += epochs;
  o = (o + 1) & ~1u;  // an instance is a whole number of 8-byte units: with one instance per extent (wide kernel, stride 1) the
                      // 64-bit queue entries of every instance stay aligned
  L.total_words = o;
  return L;
}

// Shapes with a kernel instantiation whose layout is a compile-time constant (sim_core.cuh FX): every field offset folds
// into an immediate and the extension branches the shape cannot reach are compiled out.  The host selects one only when the
// handle's layout is bit-identical to the constant and the delay model is the reference's (LogNormal served by the
// threshold table); every other handle runs the generic instantiations.
//   FX_DEFAULT4     four authors, default capacities, shared-memory queue (BASELINE configs 1-3), thread kernel
//   FX_PART7        seven authors, four partition windows, max_clock 1000, calendar queue (BASELINE configs[4]), thread
//                   kernel with 8-instance warp tiles
//   FX_COMMITTEE64  64 authors, max_clock 1000, calendar queue (BASELINE configs[3]; voting rights and silent nodes stay
//                   run-time parameters), wide kernel with 8 lanes per instance
enum : int { FX_NONE = 0, FX_DEFAULT4 = 1, FX_PART7 = 2, FX_COMMITTEE64 = 3 };
LBFT_LAYOUT_FN Layout fixed_layout(int fx) {
  return fx == FX_PART7 ? make_layout(7, 128, 512, 64, 4, 3, 1000)
                        : (fx == FX_COMMITTEE64 ? make_layout(64, 128, 32768, 512, 0, 3, 1000) : make_layout(4, 128, 64, 32, 0, 2));
}

LBFT_LAYOUT_FN uint32_t rs_table_base(const Layout& L) { return L.pay_base + L.payload_cap * L.pay_words; }
LBFT_LAYOUT_FN uint32_t res_area_base(const Layout& L, bool record_rs) {
  return rs_table_base(L) + (record_rs ? L.num_nodes * (L.round_cap + 1) : 0);
}

// One parameter set of a sweep handle (lbft_create_sweep): the values of Params below that a set replaces for the
// instances assigned to it, as HostSetup::build computed them from the set's own lbft_config.
struct SweepSet {
  double mu, sigma;
  int64_t delay_const_value;
  uint64_t uni_lo, uni_span;
  uint64_t silent_mask;
  uint32_t delay_kind, delay_const, delay_kmax;
  int32_t tci;
  uint32_t thr_off;  // first element of this set's delay thresholds in Params::sweep_thr (delay_kmax > 0)
  uint32_t tab_off;  // first element of this set's round_cap + 1 row in Params::sweep_duration / sweep_period
};

// Everything the kernel needs that is uniform over the launch.
struct Params {
  Layout L;
  uint32_t num_instances;
  int32_t max_clock;
  uint32_t delay_kind;      // LBFT_DELAY_*
  uint32_t delay_const;     // 1: sigma == 0, the LogNormal value exp(mu) was evaluated on the host
  int64_t delay_const_value;
  double mu, sigma;
  uint64_t uni_lo, uni_span;  // uniform: lo + gen_range(0..span)
  int32_t tci;                // NodeConfig.target_commit_interval (clamped to 2^30)
  uint32_t commands_per_epoch;
  uint32_t quorum;            // EpochConfiguration::quorum_threshold
  uint64_t silent_mask;
  uint32_t part_max_len;
  uint32_t record_rs;        // LBFT_FLAG_ROUND_SWITCHES: keep the DataWriter round-switch table (takes the former pad word)
  double zig_r;
  uint32_t delay_kmax;       // > 0: delay_thr[k] (k = 0..delay_kmax) is valid and replaces exp() on the device
  uint32_t pad1;
  // the voting rights travel in the parameter block itself (constant bank: no memory round trip when a vote or a
  // timeout is tallied; measured -2.3 % kernel time.  Doing the same for leader/duration/period measured slower.)
  uint32_t c_weights[64];
  // device pointers
  const uint64_t* seeds;      // [num_instances]
  const double* zig_x;        // [257]
  const double* zig_f;        // [257]
  const uint8_t* leader;      // [round_cap + 1] PacemakerState::leader(round), host-evaluated
  const int32_t* duration;    // [round_cap + 1] (delta * n^gamma) as i64, clamped to 2^30
  const int32_t* period;      // [round_cap + 1] (lambda * duration) as i64
  const uint32_t* weights;    // [num_nodes]
  const double* delay_thr;    // [delay_kmax + 1] smallest normal deviate z whose LogNormal delay is >= k (host libm)
  uint32_t* state;            // tiles
  // outputs
  uint32_t* out_commit_counts;  // [I * N]
  uint32_t* out_lc_round;       // [I * N] round of the last committed block per node
  uint64_t* out_last_state;     // [I * N]
  uint32_t* out_counters;       // [I * 12] lbft_instance_counters
  uint32_t* out_status;         // [I]
  // resumable runs (appended: nothing above moves).  The loop of this launch stops at stop_clock <= max_clock;
  // run_flags bit 0: restore the instance from its save area instead of Simulator::new
  int32_t stop_clock;
  uint32_t run_flags;
  uint32_t resumable;  // LBFT_FLAG_RESUMABLE
  uint32_t pad2;
  // appended in round 2 (nothing above moves); either may be null (host harness)
  uint32_t* out_rounds;  // [I] max over nodes of the pacemaker's active round = counters[6] (the unit of the throughput metric)
  uint32_t* out_error;   // [1] OR of the status words of every instance that ended with an error bit: the host looks at one
                         //     word instead of scanning I statuses
  // parameter sweeps (appended: nothing above moves); null / 0 on plain handles.  Only the sweep kernels read them: the
  // instance's set replaces delay_kind .. delay_const_value, mu, sigma, uni_lo, uni_span, tci, silent_mask, delay_kmax,
  // delay_thr, duration and period above.
  const SweepSet* sweep_sets;    // [num_sets]
  const uint32_t* set_of;        // [num_instances] index of each instance's set
  const double* sweep_thr;       // the sets' delay threshold tables, back to back (SweepSet::thr_off)
  const int32_t* sweep_duration; // [num_sets][round_cap + 1]
  const int32_t* sweep_period;   // [num_sets][round_cap + 1]
  uint32_t num_sets;
  uint32_t pad3;
};

}  // namespace lbft
