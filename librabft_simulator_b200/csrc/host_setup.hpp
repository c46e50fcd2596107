// host_setup.hpp — host-side preparation of a batched run: configuration validation, capacity
// selection and the tables whose arithmetic must come from the host libm so that it matches what
// the reference's Rust computes through the same libm (ln/sqrt/exp/pow), namely
//   * RandomDelay::new mu/sigma ............................. bft-lib/src/simulator.rs:99-106
//   * the rand_distr 0.4.0 ziggurat layer tables ............ (crate literals, "%.18f"-rounded)
//   * PacemakerState::leader(round) for every round ......... librabft-v2/src/pacemaker.rs:100-109
//                                                             + bft-lib/src/configuration.rs:65-75
//   * PacemakerState::duration / query-all period per n ..... librabft-v2/src/pacemaker.rs:111-124,196
// Pure C++ (no CUDA) so the CPU debugging harness in tests/hostcore can share it.  Written
// independently of oracle/ (the oracle is the checker, not a dependency).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/lbft.h"
#include "sim_params.h"

namespace lbft {

inline uint64_t host_rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }

// SipHash-1-3 (zero key) of one little-endian u64: `round.hash(&mut DefaultHasher::new())`.
inline uint64_t siphash13_u64(uint64_t mword) {
  uint64_t v0 = 0x736f6d6570736575ULL, v1 = 0x646f72616e646f6dULL, v2 = 0x6c7967656e657261ULL, v3 = 0x7465646279746573ULL;
  auto rnd = [&]() {
    v0 += v1; v1 = host_rotl(v1, 13); v1 ^= v0; v0 = host_rotl(v0, 32);
    v2 += v3; v3 = host_rotl(v3, 16); v3 ^= v2;
    v0 += v3; v3 = host_rotl(v3, 21); v3 ^= v0;
    v2 += v1; v1 = host_rotl(v1, 17); v1 ^= v2; v2 = host_rotl(v2, 32);
  };
  v3 ^= mword; rnd(); v0 ^= mword;
  uint64_t b = 8ULL << 56;
  v3 ^= b; rnd(); v0 ^= b;
  v2 ^= 0xff;
  rnd(); rnd(); rnd();
  return v0 ^ v1 ^ v2 ^ v3;
}

// EpochConfiguration::pick_author (configuration.rs:65-75): Xoshiro256** seeded through SplitMix64,
// one rand-0.8 `gen_range(0..total_votes)` (widening-multiply rejection), weighted linear scan.
inline uint32_t pick_author(const std::vector<uint32_t>& weights, uint64_t total, uint64_t seed) {
  uint64_t s[4], x = seed;
  for (int i = 0; i < 4; i++) {
    x += 0x9e3779b97f4a7c15ULL;
    uint64_t z = x;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    s[i] = z ^ (z >> 31);
  }
  uint64_t zone = (total << __builtin_clzll(total)) - 1, target;
  for (;;) {
    uint64_t v = host_rotl(s[1] * 5, 7) * 9, t = s[1] << 17;
    s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = host_rotl(s[3], 45);
    unsigned __int128 mm = (unsigned __int128)v * total;
    if ((uint64_t)mm <= zone) { target = (uint64_t)(mm >> 64); break; }
  }
  for (uint32_t a = 0; a < weights.size(); a++) {
    if (weights[a] > target) return a;
    target -= weights[a];
  }
  return 0;  // unreachable
}

inline uint32_t pow2_ceil(uint32_t v) {
  uint32_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

struct HostSetup {
  Params params{};  // pointer members are left null; the runtime fills in device addresses
  std::vector<double> zig_x, zig_f;
  std::vector<uint8_t> leader;
  std::vector<int32_t> duration, period;
  std::vector<uint32_t> weights;
  std::vector<double> delay_thr;  // see build_delay_table()
  std::string error;
  uint32_t tile_stride = 32;  // instances per state tile (lane interleaving); 1 for the warp-per-instance kernel
  bool use_wide = false;      // launch lbft_wide_kernel (one warp per instance) instead of one thread per instance
  bool wide_smem = false;     // ... with the instance state in shared memory (committees of <= 16, short horizons)
  uint32_t wide_group = 32;   // ... lanes per instance: 8 / 16 / 32

  // Parameter sweeps (lbft_create_sweep, build_sweep): the tables of every set, and each instance's set.
  std::vector<SweepSet> sets;
  std::vector<uint32_t> set_of;
  std::vector<double> sweep_thr;
  std::vector<int32_t> sweep_duration, sweep_period;

  // Events created per simulated ms, the estimate the queue mode is chosen by: ~0.14 N^2 at the reference's 10 ms mean
  // delay, proportionally more with shorter delays.
  static double event_rate(const lbft_config& c) {
    const double mean_delay = c.delay_kind == LBFT_DELAY_UNIFORM ? 0.5 * (double)(c.delay_lo + c.delay_hi) : c.delay_mean;
    return 0.14 * c.num_nodes * c.num_nodes * (10.0 / (mean_delay < 1.0 ? 1.0 : mean_delay));
  }

  bool build(const lbft_config& c) {
    if (c.struct_size != sizeof(lbft_config)) return fail("lbft_config.struct_size does not match this library (ABI mismatch)");
    if (c.num_instances == 0) return fail("num_instances must be > 0");
    if (c.num_nodes < 1 || c.num_nodes > 64) return fail("num_nodes must be in 1..64");
    if (!c.seeds) return fail("seeds must not be NULL");
    if (c.max_clock < 0 || c.max_clock >= (1 << 29)) return fail("max_clock must be in [0, 2^29)");
    if (c.flags & ~(uint32_t)(LBFT_FLAG_ROUND_SWITCHES | LBFT_FLAG_RESUMABLE | LBFT_FLAG_TRUE_DATA_SYNC)) return fail("unknown bits in flags");
    const bool tds = (c.flags & LBFT_FLAG_TRUE_DATA_SYNC) != 0;
    if (tds && (c.flags & (LBFT_FLAG_ROUND_SWITCHES | LBFT_FLAG_RESUMABLE)))
      return fail("LBFT_FLAG_TRUE_DATA_SYNC cannot be combined with recording / resumable runs");
    if (c.commands_per_epoch == 0) return fail("commands_per_epoch must be > 0");
    if (c.delta < 0 || c.target_commit_interval < 0) return fail("delta and target_commit_interval must be >= 0");
    // delta == 0 makes round durations 0: a node can then create a timeout and propose in the same update (SURVEY App.
    // C.1b), which the round-id form does not represent (the device would flag every instance LBFT_ST_INVARIANT after
    // running the whole batch).  Refuse it up front.
    if (c.delta == 0) return fail("delta = 0 is not supported: a timeout and a proposal in the same update (SURVEY App. C.1b)");
    const uint32_t N = c.num_nodes;
    Params& p = params;
    p.num_instances = c.num_instances;
    p.max_clock = (int32_t)c.max_clock;
    p.delay_kind = c.delay_kind;
    if (c.delay_kind == LBFT_DELAY_LOGNORMAL) {
      if (!(c.delay_mean > 0.0) || !(c.delay_variance >= 0.0)) return fail("LogNormal delay needs mean > 0 and variance >= 0");
      // simulator.rs:101-102
      p.mu = std::log(c.delay_mean / std::sqrt(1.0 + c.delay_variance / (c.delay_mean * c.delay_mean)));
      p.sigma = std::sqrt(std::log(1.0 + c.delay_variance / (c.delay_mean * c.delay_mean)));
      p.delay_const = p.sigma == 0.0;
      p.delay_const_value = p.delay_const ? (int64_t)std::exp(p.mu) : 0;
      if (p.delay_const && (p.delay_const_value < 0 || p.delay_const_value > (1 << 29))) return fail("constant delay out of range");
    } else if (c.delay_kind == LBFT_DELAY_UNIFORM) {
      if (c.delay_lo < 0 || c.delay_hi < c.delay_lo || c.delay_hi > (1 << 29)) return fail("uniform delay needs 0 <= lo <= hi < 2^29");
      p.uni_lo = (uint64_t)c.delay_lo;
      p.uni_span = (uint64_t)(c.delay_hi - c.delay_lo + 1);
    } else return fail("unknown delay_kind");
    p.tci = (int32_t)(c.target_commit_interval > (1 << 30) ? (1 << 30) : c.target_commit_interval);
    p.commands_per_epoch = c.commands_per_epoch > 0xffffffffULL ? 0xffffffffu : (uint32_t)c.commands_per_epoch;
    // voting rights / quorum (configuration.rs:29-56; simulated_context.rs:209-216 = all 1)
    weights.assign(N, 1);
    uint64_t total = 0;
    for (uint32_t i = 0; i < N; i++) {
      if (c.voting_rights) {
        if (c.voting_rights[i] > (1u << 24)) return fail("voting_rights entries must be <= 2^24");
        weights[i] = (uint32_t)c.voting_rights[i];
      }
      total += weights[i];
    }
    if (total == 0) return fail("total voting rights must be > 0");
    p.quorum = (uint32_t)(2 * total / 3 + 1);
    p.silent_mask = 0;
    if (c.silent)
      for (uint32_t i = 0; i < N; i++)
        if (c.silent[i]) p.silent_mask |= 1ULL << i;
    p.part_max_len = c.partition_max_len;
    if (c.partition_windows > 64) return fail("partition_windows must be <= 64");
    // capacities
    uint32_t rcap = c.round_cap ? c.round_cap : (uint32_t)(c.max_clock / 12 + 40);
    rcap = (rcap + 31) / 32 * 32;
    if (rcap < 32) rcap = 32;
    if (rcap > 32768) return fail("round_cap must be <= 32768");
    // Small committees use the scan queue (64-bit entries: time:24 | 3-kind:2 | stamp:22 | slot:8 | sender:4 |
    // receiver:4, O(1) append, linear min-scan); larger ones the binary heap with 3-word entries.
    // (explicit capacities beyond what the scan queue can encode / scan efficiently select the heap.)
    uint32_t qscan = (N <= 5 && c.max_clock < (1 << 24) - 64) ? 1u : 0u;
    if (c.payload_cap > 255 || c.queue_cap > 512) qscan = 0;
    // Kernel family.  One thread per instance needs tens of thousands of instances to fill a B200 (65 536 x 4 authors is
    // exactly one wave of warps) and serialises the 32 instances of a warp through every fan-out; one WARP per instance
    // (lbft_wide_kernel) has no cross-instance divergence, splits fan-outs, queue scans and per-author vectors over its
    // lanes, and for committees of <= 16 keeps the whole instance in shared memory.  Measured cross-over (profiles/README.md,
    // round 2): committees of <= 5 switch below ~4 K instances, larger ones always profit.  Recording / resumable handles
    // stay on the thread kernel (the wide one has no save area).  LBFT_FORCE_KERNEL=wide|thread overrides (A/B runs).
    const bool modes = (c.flags & (LBFT_FLAG_ROUND_SWITCHES | LBFT_FLAG_RESUMABLE)) != 0;
    use_wide = !modes && !tds && (N >= 6 || c.num_instances <= 4096);
    if (const char* f = std::getenv("LBFT_FORCE_KERNEL")) {
      if (!strcmp(f, "wide") && !modes && !tds) use_wide = true;
      if (!strcmp(f, "thread")) use_wide = false;
    }
    // Sparse warp tiles of the thread kernel (kernels.cuh TILE: 8 or 16 instances per warp, the other lanes retire at once):
    // the instances of a warp serialise through each other's code paths, so as long as the batch does not fill the machine
    // with full warps (2 048 warps of <= 128 registers = one wave on 148 SMs), fewer instances per warp finish sooner.
    // Measured on BASELINE configs[4] (16 384 x 7, profiles/r2j_ab_tiles.txt, r2k): 8 per warp 59.3 ms, 16 per warp 72.8, full
    // tiles 88.9, the wide kernel (8 lanes per instance) 76.2.  So for committees of 6..16 (calendar queue, plain
    // single-epoch handles): about one wave of 8-instance warps -> tile 8, of 16-instance warps -> tile 16, more -> full
    // tiles; below that the wide kernel.  LBFT_THREAD_TILE=8|16 / LBFT_FORCE_KERNEL override (A/B runs); honoured further
    // down, once the queue mode is known.
    uint32_t want_tile = 32;
    const bool env_family = std::getenv("LBFT_FORCE_KERNEL") != nullptr;
    if (const char* f = std::getenv("LBFT_THREAD_TILE")) {
      const int v = atoi(f);
      if (v == 8 || v == 16) want_tile = (uint32_t)v;
    } else if (!env_family && use_wide && N >= 6 && N <= 16 && c.max_clock <= 4095 && c.num_instances > 12288 &&
               c.commands_per_epoch >= rcap && c.queue_cap <= 0xfff0u) {
      use_wide = false;
      want_tile = c.num_instances <= 24576 ? 8u : (c.num_instances <= 49152 ? 16u : 32u);
    }
    tile_stride = use_wide ? 1u : 32u;
    // lanes per instance: enough for the committee's fan-out, few enough that a warp carries several instances
    // (measured, profiles/README.md r2e: 8 lanes per instance — four instances per warp — win once the batch fills the machine
    // with warps, committees of 64 included: 8 192 x 64 takes 1.14 s against 1.63 s with a warp per instance; below ~4 K
    // instances a whole warp per instance has the lower latency)
    wide_group = c.num_instances > 4096 ? 8u : 32u;
    if (const char* g = std::getenv("LBFT_WIDE_GROUP")) {
      const int v = atoi(g);
      if (v == 8 || v == 32) wide_group = (uint32_t)v;
    }
    // (recording round switches queues the duplicate timers the normal path elides — measured high-water marks
    // roughly double, 46 -> 64+ at N = 4 — so the smallest committees get 128 entries and the HBM scan queue)
    // (resumable runs queue them too: the event dropped at a stop must be the one the reference drops)
    const bool record = (c.flags & (LBFT_FLAG_ROUND_SWITCHES | LBFT_FLAG_RESUMABLE)) != 0;
    uint32_t qcap = c.queue_cap ? c.queue_cap : (qscan ? (N <= 4 ? (record ? 128u : 64u) : 8 * N * N) : pow2_ceil(6 * N * N + 32));
    if (2 * qcap < rcap && qscan) qcap = (rcap + 1) / 2;  // the read-out reuses the queue area as chain scratch
    if (qcap < rcap && !qscan) qcap = rcap;
    if (qcap > (1u << 20)) return fail("queue_cap too large");
    uint32_t pcap = c.payload_cap ? c.payload_cap : (N <= 4 ? 32u : (N <= 8 ? 64u : pow2_ceil(8 * N)));
    // (true data-sync keeps a snapshot per request and per response in flight as well)
    if (tds && !c.payload_cap) pcap = N <= 4 ? 128u : (N <= 8 ? 192u : 4 * pcap);
    if (pcap > 0xfff0u) return fail("payload_cap must be < 65520");
    // shortest horizons: 32-bit keys (time:14 | kind:2 | stamp:16) + 16-bit payload words, queue in shared memory
    // (16-bit stamps: ~0.14 N^2 events are created per simulated ms at the reference's 10 ms mean delay, and
    // proportionally more with shorter delays; stay well inside 65 536 — an overflow would be flagged, not silent)
    const double events_per_ms = event_rate(c);
    if (qscan && c.max_clock < (1 << 14) - 64 && qcap <= 64 && pcap <= 255 && events_per_ms * (double)c.max_clock < 32768.0)
      qscan = 2;
    // the HBM scan queue hands out 22-bit creation stamps: long horizons / very short delays go to the heap or calendar
    // queue (30-bit / 32-bit stamps) instead of aborting with LBFT_ST_QUEUE_OVERFLOW half-way through
    if (qscan == 1 && events_per_ms * (double)c.max_clock > 2.0e6) qscan = 0;
    // The wide kernel scans its (single) shared-memory queue with all 32 lanes, so the same compact entries serve committees
    // up to 16 (4-bit sender/receiver) and queues up to 1 024 entries.
    if (use_wide && N <= 16 && c.max_clock < (1 << 14) - 64 && pcap <= 255 && events_per_ms * (double)c.max_clock < 32768.0) {
      const uint32_t want = c.queue_cap ? c.queue_cap : (N <= 4 ? 64u : 8 * N * N);
      if (want <= 1024) {
        qscan = 2;
        qcap = want;
        if (2 * qcap < rcap) qcap = (rcap + 1) / 2;
      }
    }
    // everything else with a moderate horizon: calendar queue (O(1) push/pop, exact: FIFO order inside a (time, kind)
    // list is creation-stamp order); the binary heap remains for long horizons
    if (qscan == 0 && c.max_clock <= 4095 && qcap <= 0xfff0u) qscan = 3;
    // loop_until(.., Some(csv_path)) simulator.rs:380-381: keep DataWriter's round-switch table (the compile-time-layout
    // kernel never records: its layout has no table, so the generic instantiation is selected)
    p.record_rs = (c.flags & LBFT_FLAG_ROUND_SWITCHES) ? 1u : 0u;
    p.resumable = (c.flags & LBFT_FLAG_RESUMABLE) ? 1u : 0u;
    p.stop_clock = p.max_clock;
    p.run_flags = 0;
    // Epochs (node.rs:329-348): a node commits at most one command per round, so commands_per_epoch >= round_cap can never
    // be reached and the layout stays single-epoch (every BASELINE configuration).  Otherwise the per-round tables get
    // `epochs` spans of round_cap rounds each (global round id = epoch * rspan + round).
    uint32_t epochs = 1;
    if (c.commands_per_epoch < rcap) {
      if (tds) return fail("LBFT_FLAG_TRUE_DATA_SYNC needs commands_per_epoch >= round_cap (single-epoch runs)");
      wide_group = 32;
      epochs = (uint32_t)(rcap / c.commands_per_epoch) + 2;
      if (epochs > MAX_EPOCHS) epochs = MAX_EPOCHS;
      while (epochs > 2 && (uint64_t)epochs * rcap > 32768) epochs--;
      if (qcap < (epochs * rcap + 1) / 2 && qscan) qcap = (epochs * rcap + 1) / 2;  // read-out scratch (see above)
      if (qcap < epochs * rcap && !qscan) qcap = pow2_ceil(epochs * rcap);
      if (qscan == 2 && qcap > (use_wide ? 1024u : 64u)) qscan = N <= 5 ? 1u : (c.max_clock <= 4095 ? 3u : 0u);
    }
    p.L = make_layout(N, rcap, qcap, pcap, c.partition_windows, qscan, (uint32_t)c.max_clock, p.record_rs != 0, p.resumable != 0, epochs, tds);
    // (calendar queue: the sparse-tile kernels keep the occupancy words of their instances in shared memory, sim_core.cuh KS —
    // ((max_clock + 8) / 8) x tile words per warp, 14 warps per SM: horizons up to ~3 500 ms at 8 per warp, ~1 750 at 16)
    const bool ks_fits = (uint64_t)(((uint32_t)c.max_clock + 8) / 8) * want_tile <= 3584;
    if (!use_wide && want_tile != 32 && ((qscan == 3 && ks_fits && (want_tile == 8 || N <= 16)) || (qscan == 2 && want_tile == 8)) && !modes && !tds && epochs == 1)
      tile_stride = want_tile;
    // wide kernel: the whole instance lives in shared memory when the instances of 16 resident warps (32 / group each) fit on
    // an SM
    {
      const size_t bytes = sizeof(uint32_t) * (size_t)p.L.total_words + 6u * (size_t)qcap + 1024u;
      wide_smem = use_wide && qscan == 2 && epochs == 1 && bytes * (128u / wide_group) <= 56u * 1024u;
      if (const char* f = std::getenv("LBFT_WIDE_SMEM")) wide_smem = wide_smem && atoi(f) != 0;
    }
    // leader(round) for every representable round (+1: the pacemaker looks at active_round <= round_cap)
    leader.resize(rcap + 1);
    for (uint32_t r = 0; r <= rcap; r++) leader[r] = (uint8_t)pick_author(weights, total, siphash13_u64(r));
    // duration(n) = (delta as f64 * (n as f64).powf(gamma)) as i64; period = (lambda * duration as f64) as i64
    duration.resize(rcap + 1);
    period.resize(rcap + 1);
    for (uint32_t n = 0; n <= rcap; n++) {
      double dv = (double)c.delta * std::pow((double)n, c.gamma);
      int64_t dur = std::isnan(dv) ? 0 : (dv >= 9.2e18 ? INT64_MAX : (dv <= -9.2e18 ? INT64_MIN : (int64_t)dv));
      double pv = c.lambda * (double)dur;
      int64_t per = std::isnan(pv) ? 0 : (pv >= 9.2e18 ? INT64_MAX : (pv <= -9.2e18 ? INT64_MIN : (int64_t)pv));
      const int64_t CL = 1 << 30;  // any deadline beyond max_clock (< 2^29) behaves identically
      duration[n] = (int32_t)(dur > CL ? CL : (dur < -CL ? -CL : dur));
      period[n] = (int32_t)(per > CL ? CL : (per < -CL ? -CL : per));
    }
    for (uint32_t i = 0; i < 64; i++) p.c_weights[i] = i < N ? weights[i] : 0;
    build_ziggurat();
    build_delay_table();
    return true;
  }

  // A sweep handle: `c` with the values of set set_of[i] for instance i (its delay fields, target_commit_interval, delta,
  // gamma, lambda and silent are not read).  Each set is validated and its tables built by build() on the plain
  // configuration it stands for; the shared part (layout, leader table, weights, kernel family) is built once more for
  // the set with the highest event rate, with the element-wise largest queue / payload capacities of all the sets:
  // the queue modes only widen their creation stamps as the event rate grows, so no instance can raise a capacity bit
  // that its set's plain handle would not raise.
  bool build_sweep(const lbft_config& c, const lbft_param_set* ps, uint32_t num_sets, const uint32_t* set_index) {
    if (c.struct_size != sizeof(lbft_config)) return fail("lbft_config.struct_size does not match this library (ABI mismatch)");
    if (c.flags) return fail("sweep handles are plain one-shot runs: lbft_config.flags must be 0 (no recording, resumable runs or "
                             "true data-sync)");
    if (num_sets == 0 || num_sets > LBFT_MAX_PARAM_SETS) return fail("num_sets must be in 1..LBFT_MAX_PARAM_SETS");
    if (!ps || !set_index) return fail("sets and set_of_instance must not be NULL");
    for (uint32_t i = 0; i < c.num_instances; i++)
      if (set_index[i] >= num_sets) {
        char buf[128];
        snprintf(buf, sizeof buf, "set_of_instance[%u] = %u is out of range (num_sets = %u)", i, set_index[i], num_sets);
        return fail(buf);
      }
    uint8_t silent[64];
    uint32_t best = 0, qmax = 0, pmax = 0, qmin = ~0u, pmin = ~0u;
    double best_rate = -1.0;
    sets.assign(num_sets, SweepSet{});
    sweep_thr.clear();
    sweep_duration.clear();
    sweep_period.clear();
    for (uint32_t k = 0; k < num_sets; k++) {
      char pre[48];
      snprintf(pre, sizeof pre, "parameter set %u: ", k);
      if (ps[k].struct_size != sizeof(lbft_param_set)) return fail(std::string(pre) + "struct_size does not match this library (ABI mismatch)");
      if (c.num_nodes < 64 && (ps[k].silent_mask >> c.num_nodes)) return fail(std::string(pre) + "silent_mask has bits at or above num_nodes");
      const lbft_config cs = with_set(c, ps[k], silent);
      HostSetup h;
      if (!h.build(cs)) return fail(std::string(pre) + h.error);
      if (h.params.L.epochs > 1)
        return fail("sweep handles need commands_per_epoch >= round_cap (a single-epoch layout): the sweep kernels have no epoch machinery");
      const Params& q = h.params;
      SweepSet& t = sets[k];
      t.mu = q.mu; t.sigma = q.sigma; t.delay_const_value = q.delay_const_value;
      t.uni_lo = q.uni_lo; t.uni_span = q.uni_span; t.silent_mask = q.silent_mask;
      t.delay_kind = q.delay_kind; t.delay_const = q.delay_const; t.delay_kmax = q.delay_kmax; t.tci = q.tci;
      t.thr_off = (uint32_t)sweep_thr.size();
      t.tab_off = (uint32_t)sweep_duration.size();
      sweep_thr.insert(sweep_thr.end(), h.delay_thr.begin(), h.delay_thr.end());
      sweep_duration.insert(sweep_duration.end(), h.duration.begin(), h.duration.end());
      sweep_period.insert(sweep_period.end(), h.period.begin(), h.period.end());
      const double rate = event_rate(cs);
      if (rate > best_rate) { best_rate = rate; best = k; }
      qmax = std::max(qmax, q.L.queue_cap); qmin = std::min(qmin, q.L.queue_cap);
      pmax = std::max(pmax, q.L.payload_cap); pmin = std::min(pmin, q.L.payload_cap);
    }
    lbft_config cb = with_set(c, ps[best], silent);
    if (qmin != qmax) cb.queue_cap = qmax;
    if (pmin != pmax) cb.payload_cap = pmax;
    if (!build(cb)) return false;
    if (params.L.queue_cap < qmax || params.L.payload_cap < pmax) return fail("sweep capacities below a set's own (internal error)");
    // Sparse thread-kernel tiles have no sweep instantiation: those shapes run the lane-group kernel.
    if (!use_wide && tile_stride != 32) { use_wide = true; tile_stride = 1; }
    set_of.assign(set_index, set_index + c.num_instances);
    return true;
  }

  // LogNormal delay without a device-side exp(): the reference truncates exp(mu + sigma*z) to an integer
  // (simulator.rs:115-117), so only the integer part matters.  delay_thr[k] is the smallest double z with
  // (exp(mu + sigma*z) as i64) >= k, found by bisection over the doubles with the HOST libm — the very
  // function the Rust reference calls — so the device result is bit-identical to the host's by
  // construction (no last-ulp dependence on the CUDA math library).  Table: thr[0] = -inf,
  // thr[1..kmax], thr[kmax+1] = +inf, where kmax = delay at the largest deviate the ziggurat can emit.
  void build_delay_table() {
    Params& p = params;
    p.delay_kmax = 0;
    delay_thr.clear();
    if (p.delay_kind != LBFT_DELAY_LOGNORMAL || p.delay_const) return;
    const double mu = p.mu, sigma = p.sigma;
    auto D = [mu, sigma](double z) -> int64_t {
      double v = std::exp(mu + sigma * z);
      return v >= 9.0e18 ? INT64_MAX : (int64_t)v;
    };
    const double ZMAX = 14.0;  // |z| <= R + 52*ln(2)/R ~ 13.52 for the 256-layer ziggurat with 52-bit uniforms
    int64_t kmax = D(ZMAX);
    if (kmax < 1 || kmax > 4096) return;  // too wide: keep the exp() path
    auto key = [](double d) { int64_t b; memcpy(&b, &d, 8); return b < 0 ? INT64_MIN - b : b; };  // monotone map
    auto unkey = [](int64_t k) { int64_t b = k < 0 ? INT64_MIN - k : k; double d; memcpy(&d, &b, 8); return d; };
    delay_thr.assign((size_t)kmax + 2, 0.0);
    delay_thr[0] = -INFINITY;
    delay_thr[kmax + 1] = INFINITY;
    for (int64_t k = 1; k <= kmax; k++) {
      if (D(-ZMAX) >= k) { delay_thr[k] = -INFINITY; continue; }
      int64_t lo = key(-ZMAX), hi = key(ZMAX);  // D(lo) < k <= D(hi)
      while ((__int128)hi - lo > 1) {
        int64_t mid = (int64_t)(((__int128)lo + hi) >> 1);
        if (D(unkey(mid)) >= k) hi = mid; else lo = mid;
      }
      delay_thr[k] = unkey(hi);
      // exp() must be monotone across the threshold for the table to be exact: check a few ulps either side
      for (int j = 1; j <= 4; j++)
        if (D(unkey(hi + j)) < k || D(unkey(hi - j)) >= k) { delay_thr.clear(); return; }
    }
    p.delay_kmax = (uint32_t)kmax;
  }

  // rand_distr 0.4.0 ziggurat_tables.rs (ZIG_NORM_X / ZIG_NORM_F / ZIG_NORM_R): regenerated with the
  // crate's generator recurrence and passed through the "%.18f" decimal literals it ships.
  void build_ziggurat() {
    const double R = 3.6541528853610088, V = 0.00492867323399;
    std::vector<double> xs(257);
    auto f = [](double t) { return std::exp(-t * t / 2.0); };
    xs[0] = V / f(R);
    xs[1] = R;
    for (int i = 2; i < 256; i++) xs[i] = std::sqrt(-2.0 * std::log(V / xs[i - 1] + f(xs[i - 1])));
    xs[256] = 0.0;
    auto lit = [](double v) {
      char buf[64];
      snprintf(buf, sizeof buf, "%.18f", v);
      return strtod(buf, nullptr);
    };
    zig_x.resize(257);
    zig_f.resize(257);
    for (int i = 0; i <= 256; i++) {
      zig_x[i] = lit(xs[i]);
      zig_f[i] = lit(f(xs[i]));
    }
    params.zig_r = lit(R);
  }

 private:
  bool fail(const std::string& msg) {
    error = msg;
    return false;
  }
  // The plain configuration a parameter set stands for (`silent` receives the set's mask as lbft_config.silent).
  static lbft_config with_set(lbft_config c, const lbft_param_set& s, uint8_t (&silent)[64]) {
    c.delay_kind = s.delay_kind;
    c.delay_mean = s.delay_mean;
    c.delay_variance = s.delay_variance;
    c.delay_lo = s.delay_lo;
    c.delay_hi = s.delay_hi;
    c.target_commit_interval = s.target_commit_interval;
    c.delta = s.delta;
    c.gamma = s.gamma;
    c.lambda = s.lambda;
    for (uint32_t i = 0; i < 64; i++) silent[i] = (uint8_t)((s.silent_mask >> i) & 1u);
    c.silent = s.silent_mask ? silent : nullptr;
    return c;
  }
};

}  // namespace lbft
