// sim_core.cuh — the per-instance LibraBFTv2 discrete-event loop in "round-id form".
//
// One Core object simulates ONE instance (one `Simulator<NodeState<SimulatedContext>, ...>` of the
// reference) and is driven by one GPU thread; 32 instances share a warp tile (sim_params.h).  The
// code is __host__ __device__ so the same source can be compiled with g++ for CPU-side debugging
// in tests/hostcore (test infrastructure only — the product library never runs it on the host).
//
// What is restated here (reference = /root/reference, novifinancial/librabft_simulator):
//   event loop, ordering, timers, fan-out ....... bft-lib/src/simulator.rs:149-161, 200-269, 296-475
//   NodeState::update_node, commits, tracker .... librabft-v2/src/node.rs:179-202, 240-396
//   record store (verify/insert/QC/TC/3-chain) .. librabft-v2/src/record_store.rs:207-255, 257-541, 557-738
//   pacemaker ................................... librabft-v2/src/pacemaker.rs:100-124, 142-207
//   data-sync notification / request / response . librabft-v2/src/data_sync.rs:82-240
//   fake ledger (fetch/compute/commit) .......... bft-lib/src/simulated_context.rs:102-197
//   third-party arithmetic (rand 0.8.3, rand_distr 0.4.0, rand_xoshiro 0.6.0, SipHash-1-3): see
//   SURVEY.md Appendix A; restated independently of oracle/.
//
// Round-id form (SURVEY.md Appendix C, every assumption is checked at run time and raises
// LBFT_ST_INVARIANT if violated): honest leaders produce at most one block and one QC per round per
// instance, so blocks/QCs/states are identified by their round; the per-instance chain table holds
// {previous QC round, command index, proposer-local time} per round, and each node keeps three
// per-round bitsets (block known, QC known, state pending) instead of hash maps.  Request/Response
// events carry no payload because the reference answers a request on the requester itself
// (simulator.rs:446), which makes the response a no-op for the record store.
//
// Shape of the hot loop (what the SIMT hardware wants): one event per iteration; the receiving node's
// state (scalars, author masks and the 32-round window of the three per-round bitsets) is pulled
// into registers with ONE batch of independent coalesced loads, updated by branch-light code, and
// written back once; every network send of the iteration goes through ONE copy of the delay-sampling +
// enqueue code; the rare ziggurat wedge/tail and the exp() fallback live out of line.
#pragma once
#include <stdint.h>

#include <type_traits>

#include "sim_params.h"

#if defined(__CUDACC__)
#define LBFT_HD __host__ __device__ __forceinline__
#define LBFT_COLD inline __host__ __device__ __noinline__
#else
#define LBFT_HD inline
#define LBFT_COLD inline __attribute__((noinline))
#include <cmath>
#endif

// A/B switches of two exact optimisations (profiles/r2r_ab_exact.txt): see enqueue_network_event and st_u16.
#ifndef LBFT_ELIDE_SILENT
#define LBFT_ELIDE_SILENT 1
#endif
#ifndef LBFT_ST16
#define LBFT_ST16 1
#endif

namespace lbft {

// Status bits — keep in sync with include/lbft.h (static_asserted in lbft_api.cu).
enum : uint32_t {
  ST_DONE = 1u << 0,
  ST_ROUND_OVERFLOW = 1u << 1,
  ST_QUEUE_OVERFLOW = 1u << 2,
  ST_PAYLOAD_OVERFLOW = 1u << 3,
  ST_INVARIANT = 1u << 4,
  ST_EPOCH_CHANGE = 1u << 5,
  ST_DELAY_NEAR_INT = 1u << 6,
  ST_TIME_OVERFLOW = 1u << 7,
  ST_FATAL = ST_ROUND_OVERFLOW | ST_QUEUE_OVERFLOW | ST_PAYLOAD_OVERFLOW | ST_TIME_OVERFLOW,
  ST_ERROR_BITS = ST_FATAL | ST_INVARIANT  // == LBFT_ST_ERROR_MASK (static_asserted in lbft_api.cu); ST_EPOCH_CHANGE is advisory
};

constexpr int32_t NODE_TIME_NEVER = 0x7fffffff;
constexpr uint32_t PAY_NONE = 0xffffu;

// ---- small portability layer -----------------------------------------------------------------
LBFT_HD uint32_t clz32(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)__clz((int)x);
#else
  return (uint32_t)__builtin_clz(x);
#endif
}
LBFT_HD uint32_t clz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)__clzll((long long)x);
#else
  return (uint32_t)__builtin_clzll(x);
#endif
}
LBFT_HD uint32_t ctz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)(__ffsll((long long)x) - 1);
#else
  return (uint32_t)__builtin_ctzll(x);
#endif
}
LBFT_HD uint32_t ctz32(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)(__ffs((int)x) - 1);
#else
  return (uint32_t)__builtin_ctz(x);
#endif
}
LBFT_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
// IEEE double ops that must NOT be contracted into FMAs (the reference's Rust never fuses).
LBFT_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;  // host harness is built with -ffp-contract=off
#endif
}
LBFT_HD double add_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
LBFT_HD double bits_to_f64(uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)b);
#else
  double d;
  __builtin_memcpy(&d, &b, 8);
  return d;
#endif
}
LBFT_HD uint64_t rotl64(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }

// SipHash-1-3 with a zero key over a stream of u64 words (Rust DefaultHasher; the state key of
// simulated_context.rs:51-55 only ever feeds whole 8-byte integers).
struct SipWords {
  uint64_t v0, v1, v2, v3, nbytes;
  LBFT_HD SipWords() : v0(0x736f6d6570736575ULL), v1(0x646f72616e646f6dULL), v2(0x6c7967656e657261ULL), v3(0x7465646279746573ULL), nbytes(0) {}
  LBFT_HD void round() {
    v0 += v1; v1 = rotl64(v1, 13); v1 ^= v0; v0 = rotl64(v0, 32);
    v2 += v3; v3 = rotl64(v3, 16); v3 ^= v2;
    v0 += v3; v3 = rotl64(v3, 21); v3 ^= v0;
    v2 += v1; v1 = rotl64(v1, 17); v1 ^= v2; v2 = rotl64(v2, 32);
  }
  LBFT_HD void write_u64(uint64_t m) { v3 ^= m; round(); v0 ^= m; nbytes += 8; }
  LBFT_HD uint64_t finish() {
    uint64_t b = nbytes << 56;
    v3 ^= b; round(); v0 ^= b;
    v2 ^= 0xff;
    round(); round(); round();
    return v0 ^ v1 ^ v2 ^ v3;
  }
};

// View of one instance's words inside its warp tile (sim_params.h).  32-bit words are interleaved by lane
// (word w -> tile[w*STRIDE + lane]); the scan queue's 64-bit entries are interleaved at 8-byte granularity
// (entry j of the region starting at word wbase -> tile[wbase*STRIDE + j*2*STRIDE + lane*2 .. +1]), so a warp
// reading entry j issues one 256-byte coalesced access.
template <int STRIDE_>
struct TileMem {
  static constexpr int STRIDE = STRIDE_;
  uint32_t* tile;  // first word of the tile
  uint32_t lane;
  LBFT_HD uint32_t* at(uint32_t w) const { return tile + (size_t)w * STRIDE + lane; }  // then p[k * STRIDE]
  LBFT_HD uint32_t ld(uint32_t w) const { return tile[(size_t)w * STRIDE + lane]; }
  LBFT_HD void st(uint32_t w, uint32_t v) const { tile[(size_t)w * STRIDE + lane] = v; }
  LBFT_HD uint64_t* at64(uint32_t wbase) const { return reinterpret_cast<uint64_t*>(tile + (size_t)wbase * STRIDE + lane * 2); }  // then q[j * STRIDE]
};

// List of authors used for the shuffled fan-out (simulator.rs:326-343, 356-370).
template <int NMAX>
struct AuthorList;
template <>
struct AuthorList<16> {  // nibble-packed, lives in one 64-bit register
  uint64_t v = 0;
  uint32_t len = 0;
  LBFT_HD void clear() { v = 0; len = 0; }
  LBFT_HD void push(uint32_t a) { v |= (uint64_t)a << (4 * len); len++; }
  LBFT_HD uint32_t get(uint32_t i) const { return (uint32_t)(v >> (4 * i)) & 15u; }
  LBFT_HD void swap(uint32_t i, uint32_t j) {
    uint64_t d = ((v >> (4 * i)) ^ (v >> (4 * j))) & 15u;
    v ^= (d << (4 * i)) | (d << (4 * j));
  }
  LBFT_HD void fill_others(uint32_t n_nodes, uint32_t self) {  // 0..n-1 without `self`, ascending
    const uint64_t iota = 0xfedcba9876543210ULL;
    uint64_t lowmask = self ? ((1ULL << (4 * self)) - 1) : 0;
    v = (iota & lowmask) | ((iota >> 4) & ~lowmask);
    len = n_nodes - 1;
    if (len < 16) v &= (1ULL << (4 * len)) - 1;
  }
};
template <>
struct AuthorList<64> {
  uint8_t a[64];
  uint32_t len = 0;
  LBFT_HD void clear() { len = 0; }
  LBFT_HD void push(uint32_t x) { a[len++] = (uint8_t)x; }
  LBFT_HD uint32_t get(uint32_t i) const { return a[i]; }
  LBFT_HD void swap(uint32_t i, uint32_t j) { uint8_t t = a[i]; a[i] = a[j]; a[j] = t; }
  LBFT_HD void fill_others(uint32_t n_nodes, uint32_t self) {
    len = 0;
    for (uint32_t i = 0; i < n_nodes; i++)
      if (i != self) a[len++] = (uint8_t)i;
  }
};

// Per-warp shared-memory scratch of the warp-per-instance ("wide") kernel: the shuffled receiver list and the staged
// normal deviates / delays of one fan-out.
struct WideScratch {
  double z[64];
  uint16_t dly[64];
  uint8_t list[64];
};
// AuthorList with its bytes in the warp's scratch (every lane performs the same writes).
struct AuthorListShared {
  uint8_t* a;
  uint32_t len = 0;
  LBFT_HD explicit AuthorListShared(uint8_t* p) : a(p) {}
  LBFT_HD void clear() { len = 0; }
  LBFT_HD void push(uint32_t x) { a[len++] = (uint8_t)x; }
  LBFT_HD uint32_t get(uint32_t i) const { return a[i]; }
  LBFT_HD void swap(uint32_t i, uint32_t j) { uint8_t t = a[i]; a[i] = a[j]; a[j] = t; }
  LBFT_HD void fill_others(uint32_t n_nodes, uint32_t self) {
    len = 0;
    for (uint32_t i = 0; i < n_nodes; i++)
      if (i != self) a[len++] = (uint8_t)i;
  }
};

struct Actions {  // NodeUpdateActions, interfaces.rs:12-21 (should_send holds at most one author)
  int32_t next;
  int32_t send_to;
  bool broadcast, query_all;
};

// ---- out-of-line cold paths (keep the hot loop's instruction footprint small) --------------------
struct NormalSlow {
  uint64_t s0, s1, s2, s3;
  uint32_t draws;
  int32_t accepted;
  double x;
};
LBFT_HD uint64_t xoshiro_next(uint64_t& s0, uint64_t& s1, uint64_t& s2, uint64_t& s3) {
  uint64_t result = rotl64(s1 * 5, 7) * 9;
  uint64_t t = s1 << 17;
  s2 ^= s0; s3 ^= s1; s1 ^= s2; s0 ^= s3;
  s2 ^= t;
  s3 = rotl64(s3, 45);
  return result;
}
// rand_distr 0.4.0 ziggurat, the parts after the fast accept: layer-0 tail (zero_case) and wedge test.
LBFT_COLD NormalSlow normal_slow(uint64_t s0, uint64_t s1, uint64_t s2, uint64_t s3, uint32_t draws, uint32_t i, double u, double x,
                                 double f0, double f1, double zig_r) {
  NormalSlow o;
  o.accepted = 1;
  o.x = x;
  if (i == 0) {
    double xx = 1.0, yy = 0.0;
    while (mul_rn(-2.0, yy) < mul_rn(xx, xx)) {
      double a = bits_to_f64((1023ULL << 52) | (xoshiro_next(s0, s1, s2, s3) >> 12)) - (1.0 - 2.220446049250313e-16 / 2.0);  // Open01
      double b = bits_to_f64((1023ULL << 52) | (xoshiro_next(s0, s1, s2, s3) >> 12)) - (1.0 - 2.220446049250313e-16 / 2.0);
      draws += 2;
      xx = log(a) / zig_r;
      yy = log(b);
    }
    o.x = u < 0.0 ? xx - zig_r : zig_r - xx;
  } else {
    double g = mul_rn((double)(xoshiro_next(s0, s1, s2, s3) >> 11), 1.0 / 9007199254740992.0);
    draws += 1;
    double lhs = add_rn(f1, mul_rn(f0 - f1, g));
    double rhs = exp(mul_rn(-x, x) / 2.0);
    o.accepted = lhs < rhs ? 1 : 0;
  }
  o.s0 = s0; o.s1 = s1; o.s2 = s2; o.s3 = s3;
  o.draws = draws;
  return o;
}
// LogNormal delay through the device exp(): only used when no threshold table could be built.
LBFT_COLD int64_t delay_via_exp(double mu, double sigma, double z) {  // bit 62 set: near-integer advisory
  double v = exp(add_rn(mu, mul_rn(sigma, z)));
  double r = rint(v);
  int64_t flag = fabs(v - r) < 1e-9 * (r > 1.0 ? r : 1.0) ? (1LL << 62) : 0;
  if (!(v < 1.0e9)) return (1LL << 61) | 1000000000LL;
  return flag | (int64_t)v;
}

// Partition plan (EXTENSION, SURVEY App. D.3): the windows open at `clock` and the next clock at which that set changes.
// Out of line: it runs at most twice per window per run, and inlined into every send site it costs the kernels that never
// see a partition ~5 % of their code.  packed: the open windows' author masks themselves, 16 bits per window (<= 4 windows,
// <= 16 authors), instead of a bit per open window.
struct PartitionSpan {
  uint64_t open;
  int32_t until;
};
template <class Mem>
LBFT_COLD PartitionSpan partition_span(Mem m, uint32_t part_base, uint32_t windows, int32_t clock, bool packed) {
  PartitionSpan sp;
  sp.open = 0;
  sp.until = 0x7fffffff;
  for (uint32_t k = 0; k < windows; k++) {
    const int32_t t0 = (int32_t)m.ld(part_base + 4 * k), t1 = (int32_t)m.ld(part_base + 4 * k + 1);
    if (clock < t0) { if (t0 < sp.until) sp.until = t0; }
    else if (clock < t1) {
      sp.open |= packed ? (uint64_t)(m.ld(part_base + 4 * k + 2) & 0xffffu) << (16 * k) : 1ULL << k;
      if (t1 < sp.until) sp.until = t1;
    }
  }
  return sp;
}

// QMODE: 0 binary heap (3-word entries, HBM) | 1 scan queue, 64-bit keys in HBM | 2 scan queue, 32-bit keys +
// 16-bit payload words in shared memory (small committees, short horizons) | 3 calendar queue in HBM
// FX (FIXED = FX != 0): the layout is the compile-time constant fixed_layout(FX) (sim_params.h: the default four-author
// shape of BASELINE configs 1-3, the seven-author partition shape of configs[4], the 64-author shape of configs[3])
// instead of the launch parameter block: every field offset folds into an immediate.  The host only selects one for
// the reference's own delay model (LogNormal served by the threshold table), so the other delay branches — and, where
// the shape excludes them, silent nodes and partitions — are compiled out as well.
// REC: keep DataWriter's round-switch table (LBFT_FLAG_ROUND_SWITCHES, Params::record_rs).  A template parameter rather
// than a run-time test so that the non-recording instantiations carry no trace of it (the run-time test measured
// +0.8..2.0 % on the generic kernels, profiles/README.md).
// RES: resumable run (LBFT_FLAG_RESUMABLE): the loop stops at P.stop_clock the way loop_until(max_clock) does
// (simulator.rs:383-391: the first event beyond it is popped and dropped), the instance registers are saved to /
// restored from the save area, and finalize() leaves the queue alone.
// G: lanes that simulate ONE instance together.  G = 1: one thread per instance, 32 instances per warp (large batches).
// G = 8 / 16 / 32 ("wide"): a group of G lanes per instance — every lane of the group runs the same scalar state machine
// on the same values (all branches are group-uniform, so a group never diverges inside), and the data-parallel pieces
// (queue scan, per-receiver delay lookup of a fan-out, per-author vectors, table clears) are split over its lanes.  A
// warp holds 32 / G instances; they diverge from each other like the 32 instances of a thread-kernel warp do, only
// 32 / G ways.  For small batches and large committees, where one thread per instance leaves the machine empty.
// EP: the configuration can reach an epoch change (Layout::epochs > 1; node.rs:329-348).  A template parameter because the
// machinery (global round ids, per-epoch record-store reset, epoch fields of pacemaker / tracker / notification) costs ~20 %
// of the code and the instructions of a generic kernel when it is a run-time test, and no BASELINE configuration needs it.
// TDS: LBFT_FLAG_TRUE_DATA_SYNC — a data-sync request is answered by the node it was sent to, from that node's records,
// and the response's records are inserted by the requester (what data_sync.rs:183-240 is written for), instead of the
// reference simulator's dispatch to the requester itself (simulator.rs:446, SURVEY fact 5).  An opt-in NON-PARITY
// variant; plain thread-per-instance kernels only.
// KS: (QMODE 3) the calendar's kind-occupancy words live in shared memory (`km`) for the whole run instead of the instance's
// HBM block: the first hop of every pop and the occupancy test of every push become shared-memory accesses, and a push
// into an empty list issues no load at all.  Sparse-tile thread kernels and the wide kernels (a handful of instances per
// warp: (max_clock + 8) / 8 words each fit); plain one-shot runs only (nothing is kept between launches).
// SW: parameter sweep (lbft_create_sweep) — the delay model, NodeConfig (tci, duration / period tables) and silent set come
// from the instance's SweepSet (select_set, before init) instead of the launch's Params.  With SW = false nothing changes.
template <class Mem, int NMAX, int QMODE, int FX = 0, bool REC = false, bool RES = false, int G = 1, bool EP = false,
          bool TDS = false, bool KS = false, bool SW = false>
struct Core {
  static_assert(!KS || (QMODE == 3 && !RES), "shared-memory occupancy words: calendar queue, one-shot runs");
  static_assert(!(SW && (FX != FX_NONE || REC || RES || EP || TDS)), "sweeps: plain single-epoch generic kernels only");
  static constexpr bool FIXED = FX != FX_NONE;                               // compile-time layout, reference delay model
  static constexpr bool MAY_SILENT = FX == FX_NONE || FX == FX_COMMITTEE64;  // silent nodes (extension D.2) reachable
  static_assert(!(FIXED && EP), "the compile-time layout is single-epoch");
  static_assert(!(TDS && (FIXED || REC || RES || EP || G > 1)), "true data-sync: plain single-epoch thread kernels only");
  static_assert(!(FIXED && (REC || RES)), "the compile-time layout has neither a round-switch table nor a save area");
  static_assert(G == 1 || G == 8 || G == 16 || G == 32, "one thread, or a group of 8 / 16 / 32 lanes per instance");
  static_assert(G == 1 || !(REC || RES), "the wide kernel has no recording / resumable variants");
  static constexpr bool WIDE = G > 1;
  static constexpr int QS = WIDE ? 1 : 32;  // QMODE 2: stride between queue entries in shared memory (a column per lane / contiguous)
  uint32_t wl = 0;            // this thread's lane inside the group (0 when G == 1)
  uint32_t gm = 0xffffffffu;  // wide kernel: the lanes of this thread's group, as a warp mask
  WideScratch* ws = nullptr;  // wide kernel: the group's scratch
  LBFT_HD void grp_sync() const {
#if defined(__CUDA_ARCH__)
    if (WIDE) __syncwarp(gm);
#endif
  }
  // Duplicate timers are accounted at push time instead of being queued (push_timer) only when every pop does not
  // matter individually: not while recording (each pop is a sampling point) and not in resumable runs (the event
  // dropped at a stop must be the one the reference drops).
  static constexpr bool ELIDE = !(REC || RES);
  static constexpr int S = Mem::STRIDE;
  static constexpr int KSTR = WIDE ? 1 : S;  // KS: stride between this instance's occupancy words (a column per lane / contiguous)
  uint32_t* km = nullptr;                    // KS: this instance's occupancy words in shared memory
  LBFT_HD uint32_t km_ld(uint32_t w) const { return KS ? km[w * KSTR] : m.ld(L.cal_kmask + w); }
  LBFT_HD void km_st(uint32_t w, uint32_t v) const {
    if (KS) km[w * KSTR] = v;
    else m.st(L.cal_kmask + w, v);
  }
  const Params& P;
  const Layout L;
  Mem m;
  const double* zx;
  const double* zf;
  const double* thr;  // delay thresholds (shared-memory copy on the device when it fits)
  uint32_t* sk;       // QMODE 2: this lane's key column,  sk[j * 32] = time:14 | 3-kind:2 | stamp:16
  uint16_t* sd;       // QMODE 2: this lane's data column, sd[j * 32] = slot:8 | sender:4 | receiver:4
  // ---- per-instance registers ----
  uint64_t s0, s1, s2, s3;  // Xoshiro256** (simulator.rs:32)
  uint32_t draws;
  uint32_t stamp;  // Simulator.event_count / creation stamps
  uint32_t qsize;
  uint32_t status;
  int32_t clock;  // Simulator.clock
  uint32_t pay_free, pay_next;
  uint32_t proc0, proc1, proc2, proc3, cancelled, max_queue, sched_notify, dedup;
  uint32_t win;                 // bitset word index speculatively loaded with the node (hint = last node handled)
  uint32_t cal_t, cal_free, cal_next;  // QMODE 3: current bucket time, pool free list head, pool bump pointer
  int32_t part_until;  // partition plan: part_open holds for every clock below this (0: not computed yet)
  uint64_t part_open;  // ... the windows open in that span, a bit per window
  uint32_t rs_pend;  // recording only: node << 16 | active round of the round switch not yet stamped with a pop time (0: none)
  uint32_t cc0, cc1, cc2, cc3;  // chain cache: (round << 16) | previous QC round

  LBFT_HD Core(const Params& p, Mem mem, const double* zx_, const double* zf_, const double* thr_, uint32_t* sk_ = nullptr,
               uint16_t* sd_ = nullptr)
      : P(p), L(FIXED ? fixed_layout(FX) : p.L), m(mem), zx(zx_), zf(zf_), thr(thr_), sk(sk_), sd(sd_) {}

  // ------------------------------------------------------------------------------------------
  // the per-set values (SW) or the launch's (otherwise)
  // ------------------------------------------------------------------------------------------
  const SweepSet* ss = nullptr;  // SW: this instance's parameter set (read through L1; only the pointer stays in registers)
  LBFT_HD void select_set(uint32_t set) {
    ss = P.sweep_sets + set;
    thr = P.sweep_thr + ss->thr_off;
  }
#define LBFT_SET_VALUE(T, f) \
  LBFT_HD T f() const {      \
    if constexpr (SW) return ss->f; \
    else return P.f;         \
  }
  LBFT_SET_VALUE(uint32_t, delay_kind)
  LBFT_SET_VALUE(uint32_t, delay_const)
  LBFT_SET_VALUE(int64_t, delay_const_value)
  LBFT_SET_VALUE(uint32_t, delay_kmax)
  LBFT_SET_VALUE(double, mu)
  LBFT_SET_VALUE(double, sigma)
  LBFT_SET_VALUE(uint64_t, uni_lo)
  LBFT_SET_VALUE(uint64_t, uni_span)
  LBFT_SET_VALUE(int32_t, tci)
  LBFT_SET_VALUE(uint64_t, silent_mask)
#undef LBFT_SET_VALUE
  LBFT_HD int32_t round_duration(uint32_t n) const {
    if constexpr (SW) return P.sweep_duration[ss->tab_off + n];
    else return P.duration[n];
  }
  LBFT_HD int32_t round_period(uint32_t n) const {
    if constexpr (SW) return P.sweep_period[ss->tab_off + n];
    else return P.period[n];
  }

  // ------------------------------------------------------------------------------------------
  // RNG (rand_xoshiro 0.6.0 / rand 0.8.3 / rand_distr 0.4.0)
  // ------------------------------------------------------------------------------------------
  LBFT_HD void seed_rng(uint64_t seed, uint64_t& a, uint64_t& b, uint64_t& c, uint64_t& d) const {
    uint64_t x = seed, out[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      x += 0x9e3779b97f4a7c15ULL;
      uint64_t z = x;
      z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
      z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
      out[i] = z ^ (z >> 31);
    }
    a = out[0]; b = out[1]; c = out[2]; d = out[3];
  }
  LBFT_HD uint64_t next_u64() {
    draws++;
    return xoshiro_next(s0, s1, s2, s3);
  }
  LBFT_HD uint32_t gen_range_u32(uint32_t n) {  // UniformInt<u32>::sample_single_inclusive(0, n-1)
    uint32_t zone = (n << clz32(n)) - 1;
    for (;;) {
      uint32_t v = (uint32_t)(next_u64() >> 32);
      uint64_t mm = (uint64_t)v * n;
      if ((uint32_t)mm <= zone) return (uint32_t)(mm >> 32);
    }
  }
  LBFT_HD uint64_t gen_range_u64(uint64_t n) {
    uint64_t zone = (n << clz64(n)) - 1;
    for (;;) {
      uint64_t v = next_u64();
      uint64_t lo = v * n;
      if (lo <= zone) return mulhi64(v, n);
    }
  }
  LBFT_HD double standard_normal() {  // rand_distr ziggurat, 256 layers
    for (;;) {
      uint64_t bits = next_u64();
      uint32_t i = (uint32_t)bits & 0xffu;
      double u = bits_to_f64((1024ULL << 52) | (bits >> 12)) - 3.0;
      double xi = zx[i], xi1 = zx[i + 1];
      double x = mul_rn(u, xi);
      if (fabs(x) < xi1) return x;  // ~98.8 % of the draws
      NormalSlow o = normal_slow(s0, s1, s2, s3, draws, i, u, x, zf[i], zf[i + 1], P.zig_r);
      s0 = o.s0; s1 = o.s1; s2 = o.s2; s3 = o.s3;
      draws = o.draws;
      if (o.accepted) return o.x;
    }
  }
  // (exp(mu + sigma*z) as i64) == number of thresholds <= z; the thresholds were bisected on the host
  // with the host libm, so this is exact.  Any starting guess works; the walk fixes it up.
  LBFT_HD int32_t delay_from_z(double z) const {
    float g = expf((float)mu() + (float)sigma() * (float)z);
    int32_t k = g < (float)delay_kmax() ? (int32_t)g : (int32_t)delay_kmax();
    if (k < 0) k = 0;
    while (z >= thr[k + 1]) k++;
    while (z < thr[k]) k--;
    return k;
  }
  // GlobalTime::add_delay (simulator.rs:110-118): returns the delay in ms.
  LBFT_HD int32_t sample_delay() {
    if (!FIXED && delay_kind() == 1u) return (int32_t)(uni_lo() + gen_range_u64(uni_span()));
    double z = standard_normal();
    if (!FIXED && delay_const()) return (int32_t)delay_const_value();  // sigma == 0: exp(mu) evaluated by the host libm
    if (FIXED || delay_kmax()) return delay_from_z(z);
    int64_t r = delay_via_exp(mu(), sigma(), z);
    if (r & (1LL << 62)) status |= ST_DELAY_NEAR_INT;
    if (r & (1LL << 61)) status |= ST_TIME_OVERFLOW;
    return (int32_t)(r & 0x7fffffff);
  }

  // ------------------------------------------------------------------------------------------
  // memory helpers
  // ------------------------------------------------------------------------------------------
  LBFT_HD uint32_t nbase(uint32_t n) const { return L.node_base + n * L.node_words; }
  using mask_t = typename std::conditional<(NMAX > 32), uint64_t, uint32_t>::type;  // one bit per author
  LBFT_HD static mask_t ld_mask(const uint32_t* p) {
    uint64_t v = p[0];
    if (NMAX > 32) v |= (uint64_t)p[S] << 32;
    return (mask_t)v;
  }
  LBFT_HD static void st_mask(uint32_t* p, mask_t v) {
    p[0] = (uint32_t)v;
    if (NMAX > 32) p[S] = (uint32_t)((uint64_t)v >> 32);
  }
  LBFT_HD static uint32_t ld_u16(const uint32_t* p, uint32_t i) { return (p[(i >> 1) * S] >> (16 * (i & 1))) & 0xffffu; }
  // (a 16-bit store: the read-modify-write of the containing word put a dependent load — a DRAM miss in the 64-author
  // configuration — in front of every accepted timeout)
  LBFT_HD static void st_u16(uint32_t* p, uint32_t i, uint32_t v) {
    if (LBFT_ST16) {
      reinterpret_cast<uint16_t*>(p + (i >> 1) * S)[i & 1] = (uint16_t)v;  // little-endian halves, as ld_u16 reads them
      return;
    }
    uint32_t x = p[(i >> 1) * S];
    uint32_t sh = 16 * (i & 1);
    p[(i >> 1) * S] = (x & ~(0xffffu << sh)) | (v << sh);
  }
  LBFT_HD bool mbit_test(uint32_t w, uint32_t r) const { return (m.ld(w + (r >> 5)) >> (r & 31)) & 1u; }
  LBFT_HD void mbit_set(uint32_t w, uint32_t r) const { m.st(w + (r >> 5), m.ld(w + (r >> 5)) | (1u << (r & 31))); }
  // previous-QC round of block r.  The last few proposals of the instance are kept in a 4-entry direct-mapped
  // register cache (written through at propose time), which serves nearly every lookup without a dependent load.
  // (g is a GLOBAL round id, epoch * rspan + round; the value returned is the previous QC's round inside the same epoch,
  // 0 = the epoch's initial state)
  LBFT_HD uint32_t chain_prev(uint32_t g) const {
    uint32_t e = (g & 2) ? ((g & 1) ? cc3 : cc2) : ((g & 1) ? cc1 : cc0);
    if ((e >> 16) == g) return e & 0xffffu;
    return m.ld(L.chain_base + 2 * g) & 0xffffu;
  }
  // Epochs (node.rs:329-348): only configurations whose commands_per_epoch can be reached carry the machinery.
  LBFT_HD static constexpr bool multi() { return EP; }
  // GLOBAL id of the block whose state block g was executed on: its previous QC's block, or the epoch's initial state.
  LBFT_HD uint32_t chain_parent(uint32_t g) const {
    const uint32_t p = chain_prev(g);
    if (!multi()) return p;
    const uint32_t e = g / L.rspan;
    return p ? e * L.rspan + p : m.ld(L.einit_base + e);
  }
  LBFT_HD void chain_cache_put(uint32_t r, uint32_t prev) {
    uint32_t e = (r << 16) | prev;
    if ((r & 3) == 0) cc0 = e;
    if ((r & 3) == 1) cc1 = e;
    if ((r & 3) == 2) cc2 = e;
    if ((r & 3) == 3) cc3 = e;
  }

  // The receiving node's state, held in registers for the duration of one event.  Of the three per-round bitsets
  // only the 32-round word around the node's current round is cached (cw); other words go to memory.
  struct NodeRegs {
    uint32_t f[F_NSCALAR];
    mask_t vmask, tmask, tcmask;  // current_votes / current_timeouts / highest TC author sets
    uint32_t cw;                    // index of the cached bitset word
    uint32_t chb, chq, cpd;         // cached words: block known / QC known / state pending
    uint32_t dirty;                 // bit0 chb, bit1 chq, bit2 cpd modified
    uint32_t gb;                    // epoch_id * rspan: global id of this node's round 0 (0 in single-epoch layouts)
    uint32_t* nb;                   // this node's block in the tile
  };
  LBFT_HD static uint32_t epoch_of(const NodeRegs& d) { return (d.f[F_FLAGS] >> FL_EPOCH_SHIFT) & FL_EPOCH_BITS; }
  LBFT_HD void load_node(uint32_t n, NodeRegs& d) {
    uint32_t* nb = m.at(nbase(n));
    d.nb = nb;
#pragma unroll
    for (int i = 0; i < (int)F_NSCALAR; i++) d.f[i] = nb[i * S];
    d.vmask = ld_mask(nb + L.n_vmask * S);
    d.tmask = ld_mask(nb + L.n_tmask * S);
    d.tcmask = ld_mask(nb + L.n_tcmask * S);
    // speculate that this node is in the same 32-round window as the last one handled (same batch of loads)
    d.chb = nb[(L.n_hasblk + win) * S];
    d.chq = nb[(L.n_hasqc + win) * S];
    d.cpd = nb[(L.n_pend + win) * S];
    d.gb = multi() ? epoch_of(d) * L.rspan : 0u;
    uint32_t want = (d.gb + d.f[F_CUR]) >> 5;
    if (want != win) {
      d.chb = nb[(L.n_hasblk + want) * S];
      d.chq = nb[(L.n_hasqc + want) * S];
      d.cpd = nb[(L.n_pend + want) * S];
      win = want;
    }
    d.cw = want;
    d.dirty = 0;
  }
  LBFT_HD void store_node(const NodeRegs& d) const {
    uint32_t* nb = d.nb;
#pragma unroll
    for (int i = 0; i < (int)F_NSCALAR; i++) nb[i * S] = d.f[i];
    st_mask(nb + L.n_vmask * S, d.vmask);
    st_mask(nb + L.n_tmask * S, d.tmask);
    st_mask(nb + L.n_tcmask * S, d.tcmask);
    if (d.dirty & 1) nb[(L.n_hasblk + d.cw) * S] = d.chb;
    if (d.dirty & 2) nb[(L.n_hasqc + d.cw) * S] = d.chq;
    if (d.dirty & 4) nb[(L.n_pend + d.cw) * S] = d.cpd;
  }
  LBFT_HD uint32_t bword(const NodeRegs& d, uint32_t base, uint32_t cached, uint32_t r) const {
    return (r >> 5) == d.cw ? cached : d.nb[(base + (r >> 5)) * S];
  }
  // (r: a round of the node's CURRENT epoch; the bitsets are indexed by global id)
  LBFT_HD bool has_blk(const NodeRegs& d, uint32_t r) const { r += d.gb; return (bword(d, L.n_hasblk, d.chb, r) >> (r & 31)) & 1u; }
  LBFT_HD bool has_qc(const NodeRegs& d, uint32_t r) const { r += d.gb; return (bword(d, L.n_hasqc, d.chq, r) >> (r & 31)) & 1u; }
  LBFT_HD bool is_pend(const NodeRegs& d, uint32_t r) const { r += d.gb; return (bword(d, L.n_pend, d.cpd, r) >> (r & 31)) & 1u; }
  LBFT_HD void bput(NodeRegs& d, uint32_t base, uint32_t& cached, uint32_t dirty_bit, uint32_t r, bool on) const {
    uint32_t bit = 1u << (r & 31);
    if ((r >> 5) == d.cw) {
      cached = on ? (cached | bit) : (cached & ~bit);
      d.dirty |= dirty_bit;
    } else {
      uint32_t* p = d.nb + (base + (r >> 5)) * S;
      *p = on ? (*p | bit) : (*p & ~bit);
    }
  }
  LBFT_HD void set_blk(NodeRegs& d, uint32_t r) const { bput(d, L.n_hasblk, d.chb, 1u, d.gb + r, true); }
  LBFT_HD void set_qc(NodeRegs& d, uint32_t r) const { bput(d, L.n_hasqc, d.chq, 2u, d.gb + r, true); }
  LBFT_HD void set_pend(NodeRegs& d, uint32_t r, bool on) const { bput(d, L.n_pend, d.cpd, 4u, d.gb + r, on); }

  LBFT_HD static uint32_t election(const NodeRegs& d) { return (d.f[F_FLAGS] & FL_ELECTION_MASK) >> FL_ELECTION_SHIFT; }
  LBFT_HD static void set_election(NodeRegs& d, uint32_t e) { d.f[F_FLAGS] = (d.f[F_FLAGS] & ~FL_ELECTION_MASK) | (e << FL_ELECTION_SHIFT); }
  LBFT_HD static uint32_t leader_of(const NodeRegs& d) { return (d.f[F_FLAGS] >> FL_LEADER_SHIFT) & 0xffu; }

  // ------------------------------------------------------------------------------------------
  // pending-event queue, ordered by (time, 3-kind, stamp)  (simulator.rs:149-161)
  //   QMODE 1/2: unsorted array, O(1) append, linear min-scan on pop (64-bit keys in HBM / 32-bit keys in smem)
  //   QMODE 0  : binary min-heap with 3-word entries
  // ------------------------------------------------------------------------------------------
  LBFT_HD uint64_t heap_key_at(uint32_t i) const { return ((uint64_t)m.ld(L.heap_time + i) << 32) | m.ld(L.heap_key + i); }
  LBFT_HD void heap_move(uint32_t dst, uint32_t src) const {
    m.st(L.heap_time + dst, m.ld(L.heap_time + src));
    m.st(L.heap_key + dst, m.ld(L.heap_key + src));
    m.st(L.heap_data + dst, m.ld(L.heap_data + src));
  }
  // schedule_event (simulator.rs:252-264).  Events beyond max_clock can never be popped before the
  // loop ends (:389-391): they consume their creation stamp and are dropped.  Returns true if queued.
  // `data` = receiver | sender << 8 | slot << 16.
  static constexpr uint32_t kStampLimit = QMODE == 2 ? (1u << 16) : (QMODE == 1 ? (1u << 22) : (QMODE == 3 ? 0xfffffff0u : (1u << 30)));  // width of the stamp field of the queue's keys
  LBFT_HD bool push_event(int32_t time, uint32_t kind, uint32_t data) {
    uint32_t st = stamp++;
    if (stamp >= kStampLimit) status |= ST_QUEUE_OVERFLOW;
    if (time > P.max_clock) return false;
    if (qsize >= L.queue_cap) { status |= ST_QUEUE_OVERFLOW; return false; }
    if (QMODE == 3) {
      // calendar queue: one FIFO list per (time, kind).  Creation stamps grow with every push, so FIFO order inside
      // a list IS stamp order, and the pop below takes kinds in priority order: exactly (time, kind desc, stamp).
      uint32_t e;
      if (cal_free != PAY_NONE) { e = cal_free; cal_free = m.ld(L.heap_time + e); }
      else e = cal_next++;
      m.st(L.heap_key + e, data);
      const uint32_t t = (uint32_t)time, kw = t >> 3, sh = (t & 7) * 4 + kind, hw = L.cal_ht + t * 4 + kind;
      uint32_t occ = km_ld(kw);
      if ((occ >> sh) & 1) {
        uint32_t ht = m.ld(hw);
        m.st(L.heap_time + (ht >> 16), e);       // old tail -> e
        m.st(hw, (ht & 0xffffu) | (e << 16));
      } else {
        m.st(hw, e | (e << 16));
        km_st(kw, occ | (1u << sh));
      }
      qsize++;
      if (qsize > max_queue) max_queue = qsize;
      return true;
    }
    if (QMODE == 2) {
      // stamps are unique, so a 32-bit key decides every comparison; the payload word is not compared
      sk[qsize * QS] = ((uint32_t)time << 18) | ((3u - kind) << 16) | (st & 0xffffu);
      sd[qsize * QS] = (uint16_t)((((data >> 16) & 0xffu) << 8) | (((data >> 8) & 0xfu) << 4) | (data & 0xfu));
      qsize++;
      if (qsize > max_queue) max_queue = qsize;
      return true;
    }
    if (QMODE == 1) {
      // key = time:24 | 3-kind:2 | stamp:22 | slot:8 | sender:4 | receiver:4; stamps are unique, so the
      // payload bits below them never decide a comparison.
      uint64_t key = ((uint64_t)(uint32_t)time << 40) | ((uint64_t)(3u - kind) << 38) | ((uint64_t)st << 16) |
                     (uint64_t)(((data >> 16) & 0xffu) << 8) | (uint64_t)(((data >> 8) & 0xfu) << 4) | (uint64_t)(data & 0xfu);
      m.at64(L.heap_time)[(size_t)qsize * S] = key;
      qsize++;
      if (qsize > max_queue) max_queue = qsize;
      return true;
    }
    uint32_t klo = ((3u - kind) << 30) | st;
    uint64_t key = ((uint64_t)(uint32_t)time << 32) | klo;
    uint32_t i = qsize++;
    if (qsize > max_queue) max_queue = qsize;
    while (i > 0) {
      uint32_t p = (i - 1) >> 1;
      if (heap_key_at(p) <= key) break;
      heap_move(i, p);
      i = p;
    }
    m.st(L.heap_time + i, (uint32_t)time);
    m.st(L.heap_key + i, klo);
    m.st(L.heap_data + i, data);
    return true;
  }
  LBFT_HD void pop_event(int32_t& time, uint32_t& kind, uint32_t& data) {
    if (QMODE == 3) {
      // advance to the first time slot with a pending list (pushes never go below the current slot)
      uint32_t kw = cal_t >> 3;
      uint32_t occ = km_ld(kw) >> ((cal_t & 7) * 4);
      while (occ == 0) {
        cal_t = (cal_t | 7) + 1;
        kw++;
        occ = km_ld(kw);
      }
      while ((occ & 15u) == 0) { occ >>= 4; cal_t++; }
      const uint32_t nib = occ & 15u;
      kind = nib & 8u ? 3u : (nib & 4u ? 2u : (nib & 2u ? 1u : 0u));  // Timer 3 > Response 2 > Request 1 > Notify 0
      const uint32_t hw = L.cal_ht + cal_t * 4 + kind;
      const uint32_t ht = m.ld(hw), e = ht & 0xffffu;
      data = m.ld(L.heap_key + e);
      if (e == (ht >> 16)) km_st(kw, km_ld(kw) & ~(1u << ((cal_t & 7) * 4 + kind)));  // list became empty
      else m.st(hw, (ht & 0xffff0000u) | m.ld(L.heap_time + e));
      m.st(L.heap_time + e, cal_free);
      cal_free = e;
      time = (int32_t)cal_t;
      qsize--;
      return;
    }
    if (QMODE == 2 && WIDE) {
#if defined(__CUDA_ARCH__)
      // the warp scans its one queue together: lane l looks at entries l, l + 32, ...; keys are unique (creation stamps)
      __syncwarp(gm);  // entries pushed by this iteration's sends
      const uint32_t n = qsize;
      uint32_t best = 0xffffffffu, bi = 0;
      for (uint32_t j = wl; j < n; j += G) {
        const uint32_t k0 = sk[j];
        if (k0 < best) { best = k0; bi = j; }
      }
      const uint32_t mn = __reduce_min_sync(gm, best);
      const uint32_t src = (uint32_t)__ffs((int)__ballot_sync(gm, best == mn)) - 1u;  // a lane of this group (absolute index)
      bi = __shfl_sync(gm, bi, (int)src);
      const uint32_t lo = sd[bi];
      qsize = n - 1;
      __syncwarp(gm);  // everyone has read sd[bi] / its share of the keys
      if (bi != n - 1) {
        sk[bi] = sk[n - 1];
        sd[bi] = sd[n - 1];
      }
      time = (int32_t)(mn >> 18);
      kind = 3u - ((mn >> 16) & 3u);
      const uint32_t slot = lo >> 8;
      data = (lo & 0xfu) | (((lo >> 4) & 0xfu) << 8) | ((slot == 0xffu ? PAY_NONE : slot) << 16);
#endif
      return;
    }
    if (QMODE == 2) {
      uint32_t best = sk[0], bi = 0;
      const uint32_t n = qsize;
      uint32_t j = 1;
#pragma unroll 1
      for (; j + 3 < n; j += 4) {
        uint32_t k0 = sk[j * 32], k1 = sk[(j + 1) * 32], k2 = sk[(j + 2) * 32], k3 = sk[(j + 3) * 32];
        if (k0 < best) { best = k0; bi = j; }
        if (k1 < best) { best = k1; bi = j + 1; }
        if (k2 < best) { best = k2; bi = j + 2; }
        if (k3 < best) { best = k3; bi = j + 3; }
      }
#pragma unroll 1
      for (; j < n; j++) {
        uint32_t k0 = sk[j * 32];
        if (k0 < best) { best = k0; bi = j; }
      }
      uint32_t lo = sd[bi * 32];
      qsize = n - 1;
      if (bi != n - 1) {
        sk[bi * 32] = sk[(n - 1) * 32];
        sd[bi * 32] = sd[(n - 1) * 32];
      }
      time = (int32_t)(best >> 18);
      kind = 3u - ((best >> 16) & 3u);
      uint32_t slot = lo >> 8;
      data = (lo & 0xfu) | (((lo >> 4) & 0xfu) << 8) | ((slot == 0xffu ? PAY_NONE : slot) << 16);
      return;
    }
    if (QMODE == 1 && WIDE) {
#if defined(__CUDA_ARCH__)
      __syncwarp(gm);
      const uint64_t* q = m.at64(L.heap_time);
      const uint32_t n = qsize;
      uint64_t best = ~0ULL;
      uint32_t bi = 0;
      for (uint32_t j = wl; j < n; j += G) {
        const uint64_t k0 = q[(size_t)j * S];
        if (k0 < best) { best = k0; bi = j; }
      }
      // 64-bit minimum over the warp: high words first, then low words among the lanes that hold the minimal high word
      const uint32_t hi = __reduce_min_sync(gm, (uint32_t)(best >> 32));
      const uint32_t lo32 = __reduce_min_sync(gm, (uint32_t)(best >> 32) == hi ? (uint32_t)best : 0xffffffffu);
      const uint64_t mn = ((uint64_t)hi << 32) | lo32;
      const uint32_t src = (uint32_t)__ffs((int)__ballot_sync(gm, best == mn)) - 1u;
      bi = __shfl_sync(gm, bi, (int)src);
      qsize = n - 1;
      uint64_t* qw = m.at64(L.heap_time);
      const uint64_t last = qw[(size_t)(n - 1) * S];
      __syncwarp(gm);
      if (bi != n - 1) qw[(size_t)bi * S] = last;
      time = (int32_t)(mn >> 40);
      kind = 3u - ((uint32_t)(mn >> 38) & 3u);
      const uint32_t lo = (uint32_t)mn & 0xffffu, slot = lo >> 8;
      data = (lo & 0xfu) | (((lo >> 4) & 0xfu) << 8) | ((slot == 0xffu ? PAY_NONE : slot) << 16);
#endif
      return;
    }
    if (QMODE == 1) {
      // linear min-scan: independent, fully coalesced loads; no data-dependent sift chains
      const uint64_t* q = m.at64(L.heap_time);
      uint64_t best = q[0];
      uint32_t bi = 0;
      const uint32_t n = qsize;
      uint32_t j = 1;
#pragma unroll 1
      for (; j + 3 < n; j += 4) {
        uint64_t k0 = q[(size_t)j * S], k1 = q[(size_t)(j + 1) * S], k2 = q[(size_t)(j + 2) * S], k3 = q[(size_t)(j + 3) * S];
        if (k0 < best) { best = k0; bi = j; }
        if (k1 < best) { best = k1; bi = j + 1; }
        if (k2 < best) { best = k2; bi = j + 2; }
        if (k3 < best) { best = k3; bi = j + 3; }
      }
#pragma unroll 1
      for (; j < n; j++) {
        uint64_t k0 = q[(size_t)j * S];
        if (k0 < best) { best = k0; bi = j; }
      }
      qsize = n - 1;
      uint64_t* qw = m.at64(L.heap_time);
      if (bi != n - 1) qw[(size_t)bi * S] = qw[(size_t)(n - 1) * S];
      time = (int32_t)(best >> 40);
      kind = 3u - ((uint32_t)(best >> 38) & 3u);
      uint32_t lo = (uint32_t)best & 0xffffu, slot = lo >> 8;
      data = (lo & 0xfu) | (((lo >> 4) & 0xfu) << 8) | ((slot == 0xffu ? PAY_NONE : slot) << 16);
      return;
    }
    time = (int32_t)m.ld(L.heap_time);
    uint32_t klo = m.ld(L.heap_key);
    data = m.ld(L.heap_data);
    kind = 3u - (klo >> 30);
    uint32_t n = --qsize;
    if (n == 0) return;
    uint32_t lt = m.ld(L.heap_time + n), lk = m.ld(L.heap_key + n), ld_ = m.ld(L.heap_data + n);
    uint64_t key = ((uint64_t)lt << 32) | lk;
    uint32_t i = 0;
    for (;;) {
      uint32_t c = 2 * i + 1;
      if (c >= n) break;
      uint64_t kc = heap_key_at(c);
      if (c + 1 < n) {
        uint64_t kr = heap_key_at(c + 1);
        if (kr < kc) { kc = kr; c = c + 1; }
      }
      if (key <= kc) break;
      heap_move(i, c);
      i = c;
    }
    m.st(L.heap_time + i, lt);
    m.st(L.heap_key + i, lk);
    m.st(L.heap_data + i, ld_);
  }

  // notification payload pool (DataSyncNotification snapshots, shared by all receivers of one send)
  // Slot allocator.  payload_cap <= 32: a free-slot bitmask in a register (pay_free = mask of FREE slots, no memory
  // traffic); otherwise a free list threaded through word [2] of the free slots plus a bump pointer.
  // pay_next is the high-water mark of slots ever used in both cases (reported as max_payloads).
  LBFT_HD uint32_t pay_alloc() {
    uint32_t s;
    if (L.payload_cap <= 32) {
      if (pay_free == 0) { status |= ST_PAYLOAD_OVERFLOW; return PAY_NONE; }
      s = ctz32(pay_free);
      pay_free &= pay_free - 1;
      if (s >= pay_next) pay_next = s + 1;
      return s;
    }
    if (pay_free != PAY_NONE) {
      s = pay_free;
      pay_free = m.ld(L.pay_base + s * L.pay_words + 2) & 0xffffu;
    } else if (pay_next < L.payload_cap) {
      s = pay_next++;
    } else {
      status |= ST_PAYLOAD_OVERFLOW;
      s = PAY_NONE;
    }
    return s;
  }
  LBFT_HD void pay_release(uint32_t s) {
    if (L.payload_cap <= 32) { pay_free |= 1u << s; return; }
    m.st(L.pay_base + s * L.pay_words + 2, pay_free);  // link into the free list through word [2]
    pay_free = s;
  }
  LBFT_HD void pay_unref(uint32_t slot, uint32_t w2) {
    uint32_t refs = (w2 & 0xffffu) - 1;
    if (refs == 0) pay_release(slot);
    else m.st(L.pay_base + slot * L.pay_words + 2, (w2 & 0xffff0000u) | refs);
  }

  // ------------------------------------------------------------------------------------------
  // record store in round-id form
  // ------------------------------------------------------------------------------------------
  // update_current_round, record_store.rs:207-219
  LBFT_HD void update_current_round(NodeRegs& d, uint32_t round) {
    if (round <= d.f[F_CUR]) return;
    if (round >= L.rspan) { status |= ST_ROUND_OVERFLOW; return; }
    d.f[F_CUR] = round;
    d.f[F_FLAGS] &= ~(FL_PROPOSED | FL_ELECTION_MASK);
    d.tmask = 0;
    d.vmask = 0;
    d.f[F_TOW] = 0;
    d.f[F_BALLOT] = 0;
  }
  // Is the execution state of the block certified by QC `prev` (0 = the epoch's initial state)
  // available to SimulatedContext::compute?  simulated_context.rs:102-108, 128-157
  LBFT_HD bool state_available(const NodeRegs& d, uint32_t prev) const {
    if (multi()) {
      // prev == 0: the epoch's initial state — committed when the epoch began, so it is only available while it is still
      // the last committed one (simulated_context.rs:102-108; committed states leave `pending`, :163-166)
      if (prev == 0) return d.f[F_LC_ROUND] == m.ld(L.einit_base + epoch_of(d));
      return d.f[F_LC_ROUND] == d.gb + prev || is_pend(d, prev);
    }
    if (d.f[F_LC_ROUND] == prev) return true;
    if (prev == 0) return false;
    return is_pend(d, prev);
  }
  // Record::Block — verify :263-291, insert :466-476
  LBFT_HD void insert_block(NodeRegs& d, uint32_t r) {
    if (has_blk(d, r)) return;  // "Block was already inserted."
    uint32_t prev = chain_prev(d.gb + r);
    if (prev != 0 && !has_qc(d, prev)) return;  // "The previous QC (if any) must be verified first."
    // rounds are increasing by construction (the proposer's hqc round is below its current round)
    if (r == d.f[F_CUR]) d.f[F_FLAGS] |= FL_PROPOSED;  // author == leader(round) by construction (C.1)
    set_blk(d, r);
  }
  // Record::Vote — verify :292-329, insert :477-499
  LBFT_HD void insert_vote(NodeRegs& d, uint32_t r, uint32_t author) {
    if (r != d.f[F_CUR]) return;
    if (!has_blk(d, r)) return;
    if ((d.vmask >> author) & 1) return;
    d.vmask |= (mask_t)1 << author;
    if (election(d) == 0) {
      d.f[F_BALLOT] += P.c_weights[author];
      if (d.f[F_BALLOT] >= P.quorum) set_election(d, 1);
    }
  }
  // Record::QuorumCertificate — verify :330-389, insert :500-526
  LBFT_HD void insert_qc(NodeRegs& d, uint32_t r) {
    if (has_qc(d, r)) return;    // "QuorumCertificate was already inserted."
    if (!has_blk(d, r)) return;  // "The certified block hash of a QC must be verified first."
    set_qc(d, r);                // inserted before execution (:505)
    uint32_t prev = chain_prev(d.gb + r);
    if (!state_available(d, prev)) return;  // "I failed to execute a block with a QC" — QC stays in the map
    set_pend(d, r, true);
    if (r > d.f[F_HQC]) d.f[F_HQC] = r;
    update_current_round(d, r + 1);
    // update_commit_3chain_round :221-235
    if (prev != 0 && r == prev + 1 && prev - 1 > d.f[F_HCR]) {
      uint32_t r1 = chain_prev(d.gb + prev);
      if (r1 != 0 && prev == r1 + 1) {
        d.f[F_HCR] = r1;
        d.f[F_HCC] = r;
      }
    }
  }
  // Record::Timeout — verify :390-415, insert :527-538
  LBFT_HD void insert_timeout(NodeRegs& d, uint32_t round, uint32_t hcbr, uint32_t author) {
    if (hcbr > d.f[F_HQC]) return;
    if (round != d.f[F_CUR]) return;
    if ((d.tmask >> author) & 1) return;
    d.tmask |= (mask_t)1 << author;
    st_u16(d.nb + L.n_thcbr * S, author, hcbr);
    d.f[F_TOW] += P.c_weights[author];
    if (d.f[F_TOW] >= P.quorum) {
      d.tcmask = d.tmask;
      grp_sync();  // the st_u16 above is read by another lane below
      for (uint32_t i = wl; i < L.hcbr_words; i += G) d.nb[(L.n_tchcbr + i) * S] = d.nb[(L.n_thcbr + i) * S];
      grp_sync();
      d.f[F_TC_ROUND] = d.f[F_CUR];
      d.f[F_FLAGS] |= FL_HAS_TC;
      d.f[F_HTC] = d.f[F_CUR];
      update_current_round(d, d.f[F_CUR] + 1);
    }
  }
  // propose_block :655-674 (+ CommandFetcher::fetch, simulated_context.rs:116-125)
  LBFT_HD void propose_block(NodeRegs& d, uint32_t prev_round, int32_t clk) {
    uint32_t idx = d.f[F_NEXT_CMD]++;
    uint32_t r = d.f[F_CUR];
    if (idx > 0xffffu) status |= ST_ROUND_OVERFLOW;
    // App. C.1 (at most one block per round per instance) follows from C.1b, which is checked in update_node: only
    // leader(r) proposes at round r, it does so only while FL_PROPOSED is clear, and that flag is only cleared when
    // the node's round advances.  The explicit per-round "created" bitset is therefore a debug check (host harness).
#ifdef LBFT_CHECK_C1
    if (mbit_test(L.created_base, d.gb + r)) status |= ST_INVARIANT;
    mbit_set(L.created_base, d.gb + r);
#endif
    m.st(L.chain_base + 2 * (d.gb + r), prev_round | (idx << 16));
    m.st(L.chain_base + 2 * (d.gb + r) + 1, (uint32_t)clk);
    chain_cache_put(d.gb + r, prev_round);
    insert_block(d, r);
  }
  // create_vote :676-700
  LBFT_HD bool create_vote(NodeRegs& d, uint32_t n, uint32_t r, uint32_t prev) {
    if (!state_available(d, prev)) return false;
    set_pend(d, r, true);
    insert_vote(d, r, n);
    return true;
  }
  // process_commits node.rs:313-350 over committed_states_after record_store.rs:557-574 and
  // StateFinalizer::commit simulated_context.rs:161-185
  LBFT_HD void process_commits(NodeRegs& d) {
    uint32_t after = d.f[F_TRK_HCR];
    uint32_t top = d.f[F_HCC] ? d.f[F_HCR] : 0;
    while (top > after) {
      uint32_t q = top;
      for (;;) {
        uint32_t p = chain_prev(d.gb + q);
        if (p <= after) break;
        q = p;
      }
      if (!is_pend(d, q)) status |= ST_INVARIANT;  // "Committed states should be known"
      set_pend(d, q, false);
      if (chain_parent(d.gb + q) != d.f[F_LC_ROUND]) status |= ST_INVARIANT;  // happened_just_before
      d.f[F_LC_ROUND] = d.gb + q;
      d.f[F_COMMITS]++;
      after = q;
      // "check if the current epoch just ended" (node.rs:327-347): read_epoch_id = executed commands / commands_per_epoch
      // (simulated_context.rs:199-207)
      if (multi() ? d.f[F_COMMITS] / P.commands_per_epoch > epoch_of(d) : d.f[F_COMMITS] >= P.commands_per_epoch) {
        status |= ST_EPOCH_CHANGE;  // advisory: an epoch change happened in this instance
        if (!multi()) { status |= ST_ROUND_OVERFLOW; break; }  // the host sized the tables for one epoch: cannot happen
        switch_epoch(d, d.f[F_COMMITS] / P.commands_per_epoch);
        break;  // "stop delivering commits after an epoch change"
      }
    }
  }
  // node.rs:329-345: a fresh RecordStoreState for the new epoch (record_store.rs:169-198), initial state = the state just
  // committed; voting constraints reset.  past_record_stores only serves handle_request, which the simulator answers on
  // the requester itself (simulator.rs:446) with records the requester already has — nothing to keep.  The pacemaker and
  // the commit tracker notice the new epoch at their next update (pacemaker.rs:158, node.rs:372-376).
  LBFT_HD void switch_epoch(NodeRegs& d, uint32_t ne) {
    if (ne >= L.epochs) { status |= ST_ROUND_OVERFLOW; return; }
    const uint32_t init = d.f[F_LC_ROUND];
    const uint32_t seen = m.ld(L.einit_base + ne);
    if (seen != 0 && seen != init) status |= ST_INVARIANT;  // every node ends an epoch on the same block (App. C.3)
    m.st(L.einit_base + ne, init);
    store_bitset_window(d);
    d.f[F_FLAGS] = (d.f[F_FLAGS] & ~((FL_EPOCH_BITS << FL_EPOCH_SHIFT) | FL_PROPOSED | FL_ELECTION_MASK | FL_HAS_TC)) | (ne << FL_EPOCH_SHIFT);
    d.gb = ne * L.rspan;
    d.f[F_CUR] = 1;
    d.f[F_HQC] = d.f[F_HTC] = d.f[F_HCR] = d.f[F_HCC] = 0;
    d.f[F_LVR] = d.f[F_LOCKED] = 0;
    d.f[F_BALLOT] = d.f[F_TOW] = d.f[F_TC_ROUND] = 0;
    d.vmask = d.tmask = d.tcmask = 0;
    // the register window of the three bitsets moves to the new epoch's rounds
    d.cw = (d.gb + 1) >> 5;
    win = d.cw;
    d.chb = d.nb[(L.n_hasblk + d.cw) * S];
    d.chq = d.nb[(L.n_hasqc + d.cw) * S];
    d.cpd = d.nb[(L.n_pend + d.cw) * S];
  }
  LBFT_HD void store_bitset_window(NodeRegs& d) const {
    if (d.dirty & 1) d.nb[(L.n_hasblk + d.cw) * S] = d.chb;
    if (d.dirty & 2) d.nb[(L.n_hasqc + d.cw) * S] = d.chq;
    if (d.dirty & 4) d.nb[(L.n_pend + d.cw) * S] = d.cpd;
    d.dirty = 0;
  }

  // ------------------------------------------------------------------------------------------
  // NodeState::update_node, node.rs:240-304
  // ------------------------------------------------------------------------------------------
  LBFT_HD Actions update_node(uint32_t n, NodeRegs& d, int32_t clk) {
    Actions a;
    a.next = NODE_TIME_NEVER;
    a.send_to = -1;
    a.broadcast = false;
    a.query_all = false;
    // ---- Pacemaker::update_pacemaker, pacemaker.rs:142-207
    uint32_t active = (d.f[F_HQC] > d.f[F_HTC] ? d.f[F_HQC] : d.f[F_HTC]) + 1;
    // "epoch_id > self.active_epoch || (epoch_id == self.active_epoch && active_round > self.active_round)", pacemaker.rs:158
    bool new_epoch = false;
    if (multi()) {
      const uint32_t e = epoch_of(d), pe = (d.f[F_FLAGS] >> FL_PM_EPOCH_SHIFT) & FL_EPOCH_BITS;
      if (e > pe) {
        new_epoch = true;
        d.f[F_FLAGS] = (d.f[F_FLAGS] & ~(FL_EPOCH_BITS << FL_PM_EPOCH_SHIFT)) | (e << FL_PM_EPOCH_SHIFT);
      }
    }
    if (new_epoch || active > d.f[F_PMR]) {
      d.f[F_PMR] = active;
      d.f[F_PM_START] = (uint32_t)clk;
      uint32_t ld = P.leader[active];
      d.f[F_FLAGS] = (d.f[F_FLAGS] & ~(0xffu << FL_LEADER_SHIFT)) | (ld << FL_LEADER_SHIFT);
      uint32_t base = d.f[F_HCR] > 0 ? d.f[F_HCR] + 2 : 0;  // duration(), :111-124
      if (!(active > base)) { status |= ST_INVARIANT; base = active - 1; }
      d.f[F_PM_DUR] = (uint32_t)round_duration(active - base);
      d.f[F_PM_PERIOD] = (uint32_t)round_period(active - base);
      if (ld != n) a.send_to = (int32_t)ld;
    }
    const uint32_t leader = leader_of(d);
    bool propose = false, mk_timeout = false;
    bool proposed_some = d.f[F_CUR] == d.f[F_PMR] && (d.f[F_FLAGS] & FL_PROPOSED);  // proposed_block(), record_store.rs:611-634
    if (leader == n && !proposed_some) {
      propose = true;
      a.broadcast = true;
      a.next = clk;
    }
    bool has_timeout = active == d.f[F_CUR] && ((d.tmask >> n) & 1);
    if (!has_timeout) {
      int32_t deadline = (int32_t)d.f[F_PM_START] + (int32_t)d.f[F_PM_DUR];
      if (clk >= deadline) {
        mk_timeout = true;
        a.broadcast = true;
      } else if (deadline < a.next) a.next = deadline;
    } else {
      int32_t period = (int32_t)d.f[F_PM_PERIOD];
      int32_t qd = (int32_t)d.f[F_LQA] + period;
      if (clk >= qd) {
        a.query_all = true;
        qd = clk + period;
      }
      if (qd < a.next) a.next = qd;
    }
    // ---- process_pacemaker_actions, node.rs:179-202
    if (mk_timeout && propose) status |= ST_INVARIANT;  // App. C.1b
    if (mk_timeout) {
      insert_timeout(d, active, d.f[F_HQC], n);  // create_timeout, record_store.rs:636-649
      if (active > d.f[F_LVR]) d.f[F_LVR] = active;
    }
    if (propose) propose_block(d, d.f[F_HQC], clk);
    // ---- vote on the proposal, node.rs:255-276
    if (d.f[F_CUR] == d.f[F_PMR] && (d.f[F_FLAGS] & FL_PROPOSED)) {
      uint32_t r = d.f[F_CUR];
      if (r > d.f[F_LVR]) {
        uint32_t prev = chain_prev(d.gb + r);  // previous_round(), record_store.rs:588-598
        if (prev >= d.f[F_LOCKED]) {
          d.f[F_LVR] = r;
          uint32_t sp = prev ? chain_prev(d.gb + prev) : 0;  // second_previous_round(), :600-609
          if (sp > d.f[F_LOCKED]) d.f[F_LOCKED] = sp;
          if (create_vote(d, n, r, prev)) a.send_to = (int32_t)leader;
        }
      }
    }
    // ---- check_for_new_quorum_certificate (record_store.rs:702-738) and QC broadcast, node.rs:277-283
    if (election(d) == 1) {
      uint32_t r = d.f[F_CUR];
      if (P.leader[r] == n) {
        set_election(d, 2);
        // likewise at most one QC per round: the election is Closed until the round advances (debug check only)
#ifdef LBFT_CHECK_C1
        if (mbit_test(L.qcmade_base, d.gb + r)) status |= ST_INVARIANT;
        mbit_set(L.qcmade_base, d.gb + r);
#endif
        insert_qc(d, r);
        a.broadcast = true;
        a.next = clk;
      }
    }
    process_commits(d);
    // ---- CommitTracker::update_tracker, node.rs:364-396
    bool trk_new_epoch = false;
    if (multi()) {  // "if current_epoch_id > self.epoch_id", node.rs:372-376
      const uint32_t e = epoch_of(d), te = (d.f[F_FLAGS] >> FL_TRK_EPOCH_SHIFT) & FL_EPOCH_BITS;
      if (e > te) {
        trk_new_epoch = true;
        d.f[F_FLAGS] = (d.f[F_FLAGS] & ~(FL_EPOCH_BITS << FL_TRK_EPOCH_SHIFT)) | (e << FL_TRK_EPOCH_SHIFT);
      }
    }
    if (trk_new_epoch || d.f[F_HCR] > d.f[F_TRK_HCR]) {
      d.f[F_TRK_HCR] = d.f[F_HCR];
      d.f[F_TRK_TIME] = (uint32_t)clk;
    }
    int32_t tl = (int32_t)d.f[F_TRK_TIME] > (int32_t)d.f[F_LQA] ? (int32_t)d.f[F_TRK_TIME] : (int32_t)d.f[F_LQA];
    int32_t deadline = tl + tci();
    if (clk >= deadline) {
      a.query_all = true;
      deadline = clk + tci();
    }
    if (deadline < a.next) a.next = deadline;
    if (a.query_all) d.f[F_LQA] = (uint32_t)clk;
    return a;
  }

  // ------------------------------------------------------------------------------------------
  // DataSyncNode::create_notification (data_sync.rs:82-111) into a payload slot
  // ------------------------------------------------------------------------------------------
  // hcbr snapshot words (N <= 4: two words per vector) fetched BEFORE the send loop so that their latency hides
  // behind the delay sampling; measured -5.8 % kernel time.  (Prefetching the notification words before the node
  // load, by contrast, measured +9.7 % and is not done.)
  struct HcbrRegs {
    uint32_t tc[2], cur[2];
  };
  LBFT_HD void prefetch_hcbr(const NodeRegs& d, HcbrRegs& h) const {
    if (L.hcbr_words > 2) return;
    const bool has_tc = d.f[F_FLAGS] & FL_HAS_TC;
#pragma unroll
    for (uint32_t i = 0; i < 2; i++) {
      h.tc[i] = (has_tc && i < L.hcbr_words) ? d.nb[(L.n_tchcbr + i) * S] : 0u;
      h.cur[i] = (d.tmask && i < L.hcbr_words) ? d.nb[(L.n_thcbr + i) * S] : 0u;
    }
  }
  LBFT_HD void write_notification(uint32_t n, const NodeRegs& d, uint32_t slot, uint32_t refs, const HcbrRegs& h) {
    uint32_t* pb = m.at(L.pay_base + slot * L.pay_words);
    bool has_tc = d.f[F_FLAGS] & FL_HAS_TC;
    uint32_t vote = (uint32_t)((d.vmask >> n) & 1);  // current_vote(author), record_store.rs:762-764
    uint32_t prop = (d.f[F_CUR] == d.f[F_PMR] && (d.f[F_FLAGS] & FL_PROPOSED) && leader_of(d) == n) ? 1u : 0u;
    uint32_t ep = 0;
    if (multi()) {
      // proposed_block(pacemaker) is None while the pacemaker still lives in the previous epoch (record_store.rs:611-615):
      // the notification built right after an epoch change carries no proposal
      ep = epoch_of(d);
      if (((d.f[F_FLAGS] >> FL_PM_EPOCH_SHIFT) & FL_EPOCH_BITS) != ep) prop = 0;
    }
    pb[0] = d.f[F_HCC] | (d.f[F_HQC] << 16);
    pb[1 * S] = d.f[F_CUR] | ((has_tc ? d.f[F_TC_ROUND] : 0u) << 16);
    pb[2 * S] = refs | ((vote | (prop << 1)) << 16) | (ep << 18);  // [2] refcount:16 | vote | proposal | current_epoch:5
    st_mask(pb + L.p_tcmask * S, has_tc ? d.tcmask : (mask_t)0);
    st_mask(pb + L.p_curmask * S, d.tmask);
    // receivers read a timeout's highest_certified_block_round only for authors in the masks
    if (L.hcbr_words <= 2) {
#pragma unroll
      for (uint32_t i = 0; i < 2; i++) {
        if (has_tc && i < L.hcbr_words) pb[(L.p_tchcbr + i) * S] = h.tc[i];
        if (d.tmask && i < L.hcbr_words) pb[(L.p_curhcbr + i) * S] = h.cur[i];
      }
    } else {
      if (has_tc)
        for (uint32_t i = wl; i < L.hcbr_words; i += G) pb[(L.p_tchcbr + i) * S] = d.nb[(L.n_tchcbr + i) * S];
      if (d.tmask)
        for (uint32_t i = wl; i < L.hcbr_words; i += G) pb[(L.p_curhcbr + i) * S] = d.nb[(L.n_thcbr + i) * S];
      grp_sync();
    }
  }
  // DataSyncNode::handle_notification (data_sync.rs:113-177).  Returns should_sync.
  LBFT_HD bool handle_notification(NodeRegs& d, uint32_t slot, uint32_t sender) {
    uint32_t* pb = m.at(L.pay_base + slot * L.pay_words);
    uint32_t w0 = pb[0], w1 = pb[1 * S], w2 = pb[2 * S];
    mask_t tcm = ld_mask(pb + L.p_tcmask * S), curm = ld_mask(pb + L.p_curmask * S);
    uint32_t hcc = w0 & 0xffffu, hqc = w0 >> 16, cur_s = w1 & 0xffffu, tc_round = w1 >> 16;
    bool vote = (w2 >> 16) & 1, prop = (w2 >> 17) & 1;
    bool should_sync = false;
    if (multi()) {
      // Every record of a notification belongs to the sender's current epoch (data_sync.rs:82-111; quirk B.9.iii makes the
      // "previous epoch" commit certificate the current store's).  insert_network_record drops records of another epoch
      // (node.rs:150-167); a sender that is ahead makes the receiver sync (data_sync.rs:123, 131-134, 143-146).
      const uint32_t se = (w2 >> 18) & FL_EPOCH_BITS, e = epoch_of(d);
      if (se != e) {
        pay_unref(slot, w2);
        return se > e;
      }
    }
    // the two certificates, in message order: highest commit certificate, highest QC (one code copy)
#pragma unroll 1
    for (int which = 0; which < 2; which++) {
      uint32_t q = which ? hqc : hcc;
      if (q) {
        insert_qc(d, q);
        should_sync |= which ? (q > d.f[F_HQC]) : (q > d.f[F_HCR] + 2);
      }
    }
    if (prop) insert_block(d, cur_s);
    insert_timeout_groups(d, pb, tc_round, cur_s, tcm, curm);
    if (vote) insert_vote(d, cur_s, sender);
    pay_unref(slot, w2);
    return should_sync;
  }
  // timeouts of a notification / response: the TC's first, then the sender's current ones, ascending author (SURVEY B.10).
  // A group whose round is not the receiver's current round is rejected wholesale, and accepting
  // a timeout can only move the receiver's round away from the group's round.
  LBFT_HD void insert_timeout_groups(NodeRegs& d, const uint32_t* pb, uint32_t tc_round, uint32_t cur_s, mask_t tcm, mask_t curm) {
#pragma unroll 1
    for (int which = 0; which < 2; which++) {
      uint32_t round = which ? cur_s : tc_round;
      mask_t mask = which ? curm : tcm;
      if (round != 0 && round == d.f[F_CUR]) {
        const uint32_t* hp = pb + (which ? L.p_curhcbr : L.p_tchcbr) * S;
        // an author already in current_timeouts is rejected by insert_timeout whatever else holds ("already have it",
        // record_store.rs:407-411), and the set only grows while the round stands: skip them without the call
        mask &= ~d.tmask;
        while (mask) {
          uint32_t a = NMAX > 32 ? ctz64((uint64_t)mask) : ctz32((uint32_t)mask);
          mask &= mask - 1;
          insert_timeout(d, round, ld_u16(hp, a), a);
        }
      }
    }
  }

  // ------------------------------------------------------------------------------------------
  // LBFT_FLAG_TRUE_DATA_SYNC (TDS): request / response payloads in round-id form
  // ------------------------------------------------------------------------------------------
  // create_request (data_sync.rs:179-181) -> known_quorum_certificate_rounds (record_store.rs:766-799): the rounds at
  // positions 0, 1, 3, 7, ... of the QC chains that end in the highest QC and in the highest commit certificate.
  LBFT_HD void write_request_rounds(const NodeRegs& d, uint32_t slot) {
    uint32_t* pb = m.at(L.pay_base + slot * L.pay_words);
    for (uint32_t w = 0; w < L.rset_words; w++) pb[(L.p_rounds + w) * S] = 0;
#pragma unroll 1
    for (int which = 0; which < 2; which++) {
      uint32_t q = which ? d.f[F_HCC] : d.f[F_HQC];
      for (uint32_t i = 0; q != 0; i++, q = chain_prev(q))
        if ((i & (i + 1)) == 0) pb[(L.p_rounds + (q >> 5)) * S] |= 1u << (q & 31);
    }
  }
  // handle_request (data_sync.rs:183-207) on the node `n` the request was sent to -> unknown_records
  // (record_store.rs:801-831): the QCs (with their blocks) of both chains down to the first round the requester knows,
  // the timeouts (TC's, then current), the current proposed block; votes are skipped.  A snapshot, like a notification.
  LBFT_HD void write_response(uint32_t n, const NodeRegs& d, uint32_t req_slot, uint32_t slot) {
    HcbrRegs hc;
    prefetch_hcbr(d, hc);
    write_notification(n, d, slot, 1u, hc);
    uint32_t* pb = m.at(L.pay_base + slot * L.pay_words);
    const uint32_t* rq = m.at(L.pay_base + req_slot * L.pay_words);
    pb[0] = 0;  // no certificates of their own: they are in the round set
    pb[2 * S] = 1u | ((d.f[F_FLAGS] & FL_PROPOSED) ? (1u << 17) : 0u);  // current_proposed_block, whoever proposed it
    for (uint32_t w = 0; w < L.rset_words; w++) pb[(L.p_rounds + w) * S] = 0;
#pragma unroll 1
    for (int which = 0; which < 2; which++) {
      uint32_t q = which ? d.f[F_HCC] : d.f[F_HQC];
      while (q != 0 && !((rq[(L.p_rounds + (q >> 5)) * S] >> (q & 31)) & 1u)) {
        pb[(L.p_rounds + (q >> 5)) * S] |= 1u << (q & 31);
        q = chain_prev(q);
      }
    }
  }
  // handle_response (data_sync.rs:209-240): the records in order — block and QC per round ascending, timeouts, the
  // proposed block.
  LBFT_HD void handle_response(NodeRegs& d, uint32_t slot) {
    uint32_t* pb = m.at(L.pay_base + slot * L.pay_words);
    const uint32_t w1 = pb[1 * S], w2 = pb[2 * S];
    const mask_t tcm = ld_mask(pb + L.p_tcmask * S), curm = ld_mask(pb + L.p_curmask * S);
    const uint32_t cur_s = w1 & 0xffffu, tc_round = w1 >> 16;
    for (uint32_t w = 0; w < L.rset_words; w++) {
      uint32_t bits = pb[(L.p_rounds + w) * S];
      while (bits) {
        const uint32_t r = w * 32 + ctz32(bits);
        bits &= bits - 1;
        insert_block(d, r);
        insert_qc(d, r);
      }
    }
    insert_timeout_groups(d, pb, tc_round, cur_s, tcm, curm);
    if ((w2 >> 17) & 1) insert_block(d, cur_s);
    pay_unref(slot, w2);
  }

  // ------------------------------------------------------------------------------------------
  // network sends: schedule_network_event (simulator.rs:266-269) + partition drop (extension)
  // ------------------------------------------------------------------------------------------
  // The set of open windows only changes when the clock crosses a window boundary: it is recomputed then (part_until =
  // the next boundary after the clock), so a send only looks at the plan while some window is open.  Committees of <= 16
  // with <= 4 windows (BASELINE configs[4]) keep the open windows' author masks themselves in part_open, 16 bits per
  // window, and a send tests all of them at once without touching memory; otherwise part_open has a bit per open window.
  LBFT_HD bool packed_plan() const { return NMAX <= 16 && L.part_windows <= 4; }
  LBFT_HD bool partitioned(uint32_t a, uint32_t b2) {  // EXTENSION (SURVEY App. D.3)
    if (clock >= part_until) {
      const PartitionSpan sp = partition_span(m, L.part_base, L.part_windows, clock, packed_plan());
      part_open = sp.open;
      part_until = sp.until;
    }
    if (packed_plan()) return (((part_open >> a) ^ (part_open >> b2)) & 0x0001000100010001ULL) != 0;
    for (uint64_t open = part_open; open; open &= open - 1) {
      const uint32_t k = ctz64(open);
      uint64_t mask = m.ld(L.part_base + 4 * k + 2) | ((uint64_t)m.ld(L.part_base + 4 * k + 3) << 32);
      if (((mask >> a) ^ (mask >> b2)) & 1) return true;
    }
    return false;
  }
  LBFT_HD bool schedule_network_event(uint32_t kind, uint32_t receiver, uint32_t sender, uint32_t slot) {
    return enqueue_network_event(kind, receiver, sender, slot, sample_delay());
  }
  LBFT_HD bool enqueue_network_event(uint32_t kind, uint32_t receiver, uint32_t sender, uint32_t slot, int32_t delay) {
    int32_t t = clock + delay;
    if (L.part_windows && partitioned(receiver, sender)) {
      stamp++;
      return false;
    }
    // EXTENSION D.2, exact elision: a notification addressed to a silent node, or a request whose addressee is silent, is
    // dropped by the loop right after its pop with no effect but the event counters (run(): the clock it advances is
    // overwritten by the next live event before anything reads it).  Account for the pop here — it is certain: every queued
    // event up to max_clock is popped before a one-shot run ends — and keep the event, a third of the 64-author
    // configuration's traffic, out of the queue and out of the snapshot's reference count.  It still takes its creation
    // stamp and its delay draw.  Not while recording / resumable / true-data-sync (every pop is observable there).
    if (LBFT_ELIDE_SILENT && ELIDE && !TDS && MAY_SILENT && silent_mask() && kind != EV_RESPONSE &&
        ((silent_mask() >> (kind == EV_NOTIFY ? receiver : sender)) & 1)) {
      stamp++;
      if (stamp >= kStampLimit) status |= ST_QUEUE_OVERFLOW;
      if (t <= P.max_clock) {
        if (kind == EV_NOTIFY) proc0++;
        else proc1++;
      }
      return false;
    }
    return push_event(t, kind, receiver | (sender << 8) | (slot << 16));
  }
  template <bool W = WIDE>
  LBFT_HD typename std::enable_if<W, AuthorListShared>::type make_list() const { return AuthorListShared(ws->list); }
  template <bool W = WIDE>
  LBFT_HD typename std::enable_if<!W, AuthorList<(NMAX <= 16 ? 16 : 64)>>::type make_list() const { return AuthorList<(NMAX <= 16 ? 16 : 64)>(); }
  LBFT_HD void push_timer(uint32_t n, NodeRegs& d, int32_t t) {
    // (not while recording round switches: every pop is a DataWriter sampling point, data_writer.rs:34-50, so the
    // duplicate has to be popped where the reference pops it)
    if (ELIDE && (uint32_t)t == d.f[F_LAST_TIMER]) {
      // An UpdateTimerEvent for (n, t) is already pending with a smaller stamp.  The duplicate could
      // only ever be popped right after it (same time) and be cancelled by
      // ignore_scheduled_updates_until (simulator.rs:403-410) with no side effect: account for it
      // as popped+cancelled now and do not queue it (SURVEY App. C.4).
      stamp++;
      if (t <= P.max_clock) { proc3++; cancelled++; dedup++; }
      return;
    }
    d.f[F_LAST_TIMER] = (uint32_t)t;
    push_event(t, EV_TIMER, n | (n << 8) | (PAY_NONE << 16));
  }

  // ------------------------------------------------------------------------------------------
  // Simulator::new, simulator.rs:200-250 (+ make_initial_state node.rs:87-114, record_store.rs:169-198)
  // ------------------------------------------------------------------------------------------
  LBFT_HD void init(uint64_t seed) {
    const uint32_t N = L.num_nodes;
    seed_rng(seed, s0, s1, s2, s3);
    draws = 0; stamp = 0; qsize = 0; status = 0; clock = 0;
    pay_free = L.payload_cap <= 32 ? (L.payload_cap == 32 ? 0xffffffffu : ((1u << L.payload_cap) - 1)) : PAY_NONE;
    pay_next = 0;
    proc0 = proc1 = proc2 = proc3 = cancelled = max_queue = sched_notify = dedup = 0;
    win = 0;
    cc0 = cc1 = cc2 = cc3 = 0;
    cal_t = 0; cal_free = PAY_NONE; cal_next = 0;
    part_until = 0; part_open = 0;
    if (REC) {
      rs_pend = 0;
      for (uint32_t w = 0; w < N * (L.round_cap + 1); w++) m.st(rs_table_base(L) + w, 0);
    }
    // (table clears are split over the lanes of the group; G == 1: wl == 0, the plain loops)
    if (QMODE == 3)
      for (uint32_t w = wl; w < (L.cal_times + 7) / 8; w += G) km_st(w, 0);
    for (uint32_t w = wl; w < N * L.node_words; w += G) m.st(L.node_base + w, 0);
    for (uint32_t w = wl; w < 2 * L.rset_words; w += G) m.st(L.created_base + w, 0);
    if (multi())
      for (uint32_t w = wl; w < L.epochs; w += G) m.st(L.einit_base + w, 0);
    grp_sync();
    // EXTENSION D.3: partition plan from a separate stream; must match oracle_capi.cpp make_partition_plan
    if (L.part_windows) {
      uint64_t k0 = s0, k1 = s1, k2 = s2, k3 = s3;
      uint32_t kd = draws;
      seed_rng(seed ^ 0xD1B54A32D192ED03ULL, s0, s1, s2, s3);
      uint64_t nsub = N >= 64 ? 0xfffffffffffffffeULL : ((1ULL << N) - 2);
      for (uint32_t k = 0; k < L.part_windows; k++) {
        int64_t t0 = (int64_t)gen_range_u64((uint64_t)P.max_clock + 1);
        int64_t len = 1 + (int64_t)gen_range_u64(P.part_max_len ? P.part_max_len : 1);
        uint64_t mask = N >= 2 ? 1 + gen_range_u64(nsub) : 0;
        m.st(L.part_base + 4 * k, (uint32_t)t0);
        m.st(L.part_base + 4 * k + 1, (uint32_t)(t0 + len));
        m.st(L.part_base + 4 * k + 2, (uint32_t)mask);
        m.st(L.part_base + 4 * k + 3, (uint32_t)(mask >> 32));
      }
      s0 = k0; s1 = k1; s2 = k2; s3 = k3;
      draws = kd;
    }
#pragma unroll 1
    for (uint32_t n = 0; n < N; n++) {
      int32_t startup = sample_delay() + 1;
      uint32_t b = nbase(n);
      m.st(b + F_STARTUP, (uint32_t)startup);
      m.st(b + F_IGNORE, (uint32_t)(startup - 1));
      m.st(b + F_CUR, 1);
      m.st(b + F_FLAGS, FL_LEADER_NONE << FL_LEADER_SHIFT);
      m.st(b + F_LAST_TIMER, (uint32_t)startup);
      push_event(startup, EV_TIMER, n | (n << 8) | (PAY_NONE << 16));
    }
  }

  // ------------------------------------------------------------------------------------------
  // Simulator::loop_until, simulator.rs:380-475, with process_node_actions (:296-378) folded in
  // ------------------------------------------------------------------------------------------
  LBFT_HD void run() {
    const uint32_t N = L.num_nodes;
#pragma unroll 1
    while (qsize > 0 && !(status & ST_FATAL)) {
      int32_t t;
      uint32_t kind, data;
      pop_event(t, kind, data);
      // one-shot runs: unreachable, such events are dropped at push.  Resumable runs: loop_until's own exit,
      // simulator.rs:389-391 — the popped event is gone.
      if (t > (RES ? P.stop_clock : P.max_clock)) {
        // the dropped event owned a reference to its notification snapshot: give it back, or every stop leaks a slot
        if (RES && kind == EV_NOTIFY && (data >> 16) != PAY_NONE)
          pay_unref(data >> 16, m.ld(L.pay_base + (data >> 16) * L.pay_words + 2));
        break;
      }
      // DataWriter::update_round_number (data_writer.rs:34-50), called at simulator.rs:393-394 with the popped event's
      // own scheduled time.  Only the node that handled the previous event can have a larger active round than at
      // the previous pop, so at most one switch is pending.
      if (REC && rs_pend) {
        const uint32_t rn = rs_pend >> 16, rr = rs_pend & 0xffffu;
        // slot [node][0] holds DataWriter::max_round_per_node (round 0 itself is never recorded: 0 > 0 is false): after an
        // epoch change the active round restarts at 1 and only rounds beyond the recorded maximum count (data_writer.rs:43-46)
        const uint32_t row = rs_table_base(L) + rn * (L.round_cap + 1);
        if (rr <= L.round_cap && rr > m.ld(row)) {
          m.st(row + rr, (uint32_t)t + 1u);
          m.st(row, rr);
        }
        rs_pend = 0;
      }
      if (t > clock) clock = t;
      const uint32_t receiver = data & 0xffu, sender = (data >> 8) & 0xffu, slot = data >> 16;
      proc0 += kind == EV_NOTIFY;
      proc1 += kind == EV_REQUEST;
      proc2 += kind == EV_RESPONSE;
      proc3 += kind == EV_TIMER;
      // EXTENSION D.2: silent nodes handle nothing and answer no request
      if (MAY_SILENT && silent_mask()) {
        bool drop = (silent_mask() >> receiver) & 1;
        if (kind == EV_REQUEST && ((silent_mask() >> sender) & 1)) drop = true;
        if (drop) {
          if (kind == EV_NOTIFY || (TDS && slot != PAY_NONE)) pay_unref(slot, m.ld(L.pay_base + slot * L.pay_words + 2));
          continue;
        }
      }
      NodeRegs d;
      Actions a;
      a.next = NODE_TIME_NEVER;
      a.send_to = -1;
      a.broadcast = false;
      a.query_all = false;
      bool should_sync = false;
      uint32_t sync_slot = PAY_NONE;  // TDS: the sync request's payload, written when handle_notification asks for it
      const bool is_request = kind == EV_REQUEST;  // answered by `receiver` itself (simulator.rs:446): no state change
      if (TDS && is_request) load_node(sender, d);  // ... unless the node it was sent to answers (read only, never stored)
      if (!is_request) {
        load_node(receiver, d);
        const uint32_t pmr_before = d.f[F_PMR];
        if (kind == EV_TIMER && clock <= (int32_t)d.f[F_IGNORE]) {
          cancelled++;
          continue;
        }
        if (kind == EV_NOTIFY) {
          should_sync = handle_notification(d, slot, sender);
          if (TDS && should_sync) {  // create_request_internal runs inside handle_notification, before the update (data_sync.rs:172-176)
            sync_slot = pay_alloc();
            if (sync_slot != PAY_NONE) write_request_rounds(d, sync_slot);
          }
        }
        if (TDS && kind == EV_RESPONSE && slot != PAY_NONE) handle_response(d, slot);
        a = update_node(receiver, d, clock - (int32_t)d.f[F_STARTUP]);
        if (REC && d.f[F_PMR] > pmr_before) rs_pend = (receiver << 16) | (d.f[F_PMR] & 0xffffu);
        // next UpdateTimerEvent, simulator.rs:311-324
        int64_t from_node = a.next == NODE_TIME_NEVER ? (int64_t)0x7fffffff : (int64_t)a.next + (int32_t)d.f[F_STARTUP];
        int64_t nt = from_node > (int64_t)clock + 1 ? from_node : (int64_t)clock + 1;
        if (nt > 0x7ffffff0) nt = 0x7ffffff0;
        d.f[F_IGNORE] = (uint32_t)((int32_t)nt - 1);
      }
      // All the network sends of this event go through ONE copy of the sampling + enqueue code, in the reference's
      // RNG / creation-stamp order: [sync request (simulator.rs:427-433)] -> timer stamp (:311-324) ->
      // shuffle(receivers), notifications (:326-354) -> shuffle(senders), requests (:356-377); a Request event
      // only schedules its Response (:448-452).  The 32 instances of a warp execute the passes together, so the
      // cost of an iteration is the number of passes x the longest list in each.  Two exact foldings keep that
      // small: a Request event's single Response send, and a query-all fan-out whose notification list is empty,
      // run inside the notification pass (nothing of the same instance lies between them in the RNG stream).
      typename std::conditional<WIDE, AuthorListShared, AuthorList<(NMAX <= 16 ? 16 : 64)>>::type list = make_list();
      bool query_pending = a.query_all;
      // (a lane only enters the passes it has something to do in: pass 0 when it owes a sync request, pass 2 when a
      // query-all is still pending after pass 1)
#pragma unroll 1
      for (int phase = should_sync ? 0 : 1; phase < 2 || (phase == 2 && query_pending); phase++) {
        uint32_t ev_kind = EV_REQUEST, pslot = PAY_NONE;
        bool to_other = false;  // notifications travel to `other`; requests/responses are addressed to the node itself
        list.clear();
        if (phase == 0) {
          if (should_sync) list.push(sender);
        } else if (phase == 1) {
          if (is_request) {
            ev_kind = EV_RESPONSE;
            list.push(sender);
          } else {
            push_timer(receiver, d, (int32_t)d.f[F_IGNORE] + 1);  // its stamp comes after the sync request, before the fan-out
            if (a.broadcast) list.fill_others(N, receiver);
            else if (a.send_to >= 0 && (uint32_t)a.send_to != receiver) list.push((uint32_t)a.send_to);
            if (list.len) {
              ev_kind = EV_NOTIFY;
              to_other = true;
            } else if (query_pending) {
              list.fill_others(N, receiver);
              query_pending = false;
            }
          }
        } else {
          if (query_pending) list.fill_others(N, receiver);
        }
        for (uint32_t i = list.len; i-- > 1;) list.swap(i, gen_range_u32(i + 1));  // SliceRandom::shuffle
        if (list.len == 0) continue;
        HcbrRegs hc;
        if (to_other) {
          pslot = pay_alloc();
          sched_notify += list.len;
          prefetch_hcbr(d, hc);
        }
        const bool req_payload = TDS && ev_kind == EV_REQUEST, resp_payload = TDS && ev_kind == EV_RESPONSE;
        if (req_payload) {
          pslot = phase == 0 ? sync_slot : pay_alloc();
          if (phase != 0 && pslot != PAY_NONE) write_request_rounds(d, pslot);  // create_request at send time, simulator.rs:365-368
        }
        if (resp_payload) pslot = pay_alloc();
        uint32_t queued = 0;
        // Wide kernel, table-served LogNormal delay: the normal deviates of the fan-out are drawn first (the RNG stream is
        // sequential), then each lane turns its share of them into delays, then the events are queued in list order.
        // Nothing else draws from the stream or takes a creation stamp in between, so the order of both is unchanged.
        const bool staged = WIDE && list.len > 1 && (FIXED || (delay_kind() == 0u && !delay_const() && delay_kmax() != 0));
        if (staged) {
          for (uint32_t i = 0; i < list.len; i++) ws->z[i] = standard_normal();
          grp_sync();
          for (uint32_t i = wl; i < list.len; i += G) ws->dly[i] = (uint16_t)delay_from_z(ws->z[i]);
          grp_sync();
        }
#pragma unroll 1
        for (uint32_t i = 0; i < list.len; i++) {
          uint32_t other = list.get(i);
          uint32_t ev_recv = to_other ? other : receiver, ev_send = to_other ? receiver : other;
          if (staged ? enqueue_network_event(ev_kind, ev_recv, ev_send, pslot, (int32_t)ws->dly[i])
                     : schedule_network_event(ev_kind, ev_recv, ev_send, pslot)) queued++;
        }
        if (to_other && pslot != PAY_NONE) {
          if (queued) write_notification(receiver, d, pslot, queued, hc);
          else pay_release(pslot);
        }
        if (req_payload && pslot != PAY_NONE) {
          if (queued) m.st(L.pay_base + pslot * L.pay_words + 2, queued);  // one reference per queued copy of the request
          else pay_release(pslot);
        }
        if (resp_payload) {
          if (pslot != PAY_NONE) {
            if (queued && slot != PAY_NONE) write_response(sender, d, slot, pslot);
            else pay_release(pslot);
          }
          if (slot != PAY_NONE) pay_unref(slot, m.ld(L.pay_base + slot * L.pay_words + 2));  // this copy of the request has been answered
        }
      }
      if (!is_request) store_node(d);
    }
    if (!(status & ST_FATAL)) status |= ST_DONE;
  }

  // ------------------------------------------------------------------------------------------
  // read-out: commit counts, last committed round and state key per node; counters; status
  // ------------------------------------------------------------------------------------------
  // ------------------------------------------------------------------------------------------
  // Resumable runs: the per-instance registers (and, QMODE 2, the shared-memory queue) between two launches
  // ------------------------------------------------------------------------------------------
  LBFT_HD void save_regs() {
    const uint32_t b = res_area_base(L, REC);
    uint32_t w = b;
    const uint64_t sx[4] = {s0, s1, s2, s3};
    for (int i = 0; i < 4; i++) { m.st(w++, (uint32_t)sx[i]); m.st(w++, (uint32_t)(sx[i] >> 32)); }
    const uint32_t r[] = {draws, stamp, qsize, status, (uint32_t)clock, pay_free, pay_next, proc0, proc1, proc2, proc3, cancelled,
                          max_queue, sched_notify, dedup, win, cal_t, cal_free, cal_next, REC ? rs_pend : 0u, cc0, cc1, cc2, cc3};
    static_assert(8 + sizeof(r) / 4 <= RES_REG_WORDS, "save area too small");
    for (uint32_t i = 0; i < sizeof(r) / 4; i++) m.st(w++, r[i]);
    if (QMODE == 2) {
      const uint32_t q = b + RES_REG_WORDS + L.round_cap, qd = q + L.queue_cap;
      for (uint32_t j = 0; j < qsize; j++) m.st(q + j, sk[j * 32]);
      for (uint32_t j = 0; j < qsize; j += 2) m.st(qd + (j >> 1), (uint32_t)sd[j * 32] | (j + 1 < qsize ? (uint32_t)sd[(j + 1) * 32] << 16 : 0u));
    }
  }
  LBFT_HD void restore_regs() {
    const uint32_t b = res_area_base(L, REC);
    uint32_t w = b;
    part_until = 0; part_open = 0;  // recomputed at the first send
    uint64_t sx[4];
    for (int i = 0; i < 4; i++) { uint64_t lo = m.ld(w++); uint64_t hi = m.ld(w++); sx[i] = lo | (hi << 32); }
    s0 = sx[0]; s1 = sx[1]; s2 = sx[2]; s3 = sx[3];
    draws = m.ld(w++); stamp = m.ld(w++); qsize = m.ld(w++); status = m.ld(w++); clock = (int32_t)m.ld(w++);
    pay_free = m.ld(w++); pay_next = m.ld(w++); proc0 = m.ld(w++); proc1 = m.ld(w++); proc2 = m.ld(w++); proc3 = m.ld(w++);
    cancelled = m.ld(w++); max_queue = m.ld(w++); sched_notify = m.ld(w++); dedup = m.ld(w++); win = m.ld(w++);
    cal_t = m.ld(w++); cal_free = m.ld(w++); cal_next = m.ld(w++);
    const uint32_t rp = m.ld(w++);
    if (REC) rs_pend = rp;
    cc0 = m.ld(w++); cc1 = m.ld(w++); cc2 = m.ld(w++); cc3 = m.ld(w++);
    if (QMODE == 2) {
      const uint32_t q = b + RES_REG_WORDS + L.round_cap, qd = q + L.queue_cap;
      for (uint32_t j = 0; j < qsize; j++) {
        sk[j * 32] = m.ld(q + j);
        sd[j * 32] = (uint16_t)(m.ld(qd + (j >> 1)) >> ((j & 1) * 16));
      }
    }
  }

  LBFT_HD void finalize(uint32_t inst) {
    const uint32_t N = L.num_nodes;
    const uint32_t scratch = RES ? res_area_base(L, REC) + RES_REG_WORDS : L.heap_time;
    uint32_t max_round = 0;
    for (uint32_t n = 0; n < N; n++) {
      uint32_t b = nbase(n);
      uint32_t commits = m.ld(b + F_COMMITS), lc = m.ld(b + F_LC_ROUND), pmr = m.ld(b + F_PMR);
      if (pmr > max_round) max_round = pmr;
      // lay the chain out in commit order in the (now dead) event queue area, then hash it:
      // SimulatedLedgerState::key, simulated_context.rs:51-55
      uint32_t depth = 0;
      for (uint32_t r = lc; r != 0; r = chain_parent(r)) depth++;
      if (depth != commits) status |= ST_INVARIANT;
      uint32_t i = depth;
      for (uint32_t r = lc; r != 0 && i > 0; r = chain_parent(r)) m.st(scratch + (--i), r);
      SipWords h;
      h.write_u64(depth);
      for (uint32_t k = 0; k < depth; k++) {
        uint32_t r = m.ld(scratch + k);
        uint32_t c0 = m.ld(L.chain_base + 2 * r);
        int32_t tm = (int32_t)m.ld(L.chain_base + 2 * r + 1);
        h.write_u64(P.leader[multi() ? r % L.rspan : r]);
        h.write_u64(c0 >> 16);
        h.write_u64((uint64_t)(int64_t)tm);
      }
      P.out_commit_counts[(size_t)inst * N + n] = commits;
      P.out_lc_round[(size_t)inst * N + n] = lc;
      P.out_last_state[(size_t)inst * N + n] = h.finish();
    }
    uint32_t* c = P.out_counters + (size_t)inst * 12;
    c[0] = proc0; c[1] = proc1; c[2] = proc2; c[3] = proc3;
    c[4] = cancelled; c[5] = stamp; c[6] = max_round; c[7] = draws; c[8] = max_queue;
    c[9] = sched_notify; c[10] = pay_next; c[11] = dedup;
    P.out_status[inst] = status;
    if (P.out_rounds) P.out_rounds[inst] = max_round;
    if (P.out_error && (status & ST_ERROR_BITS)) {
#if defined(__CUDA_ARCH__)
      atomicOr(P.out_error, status);
#else
      *P.out_error |= status;
#endif
    }
  }
};

}  // namespace lbft
