/* lbft.h — C ABI of the B200-native batched LibraBFTv2 discrete-event simulator.
 *
 * Drop-in boundary for the ONE hot path of novifinancial/librabft_simulator (reference checkout
 * /root/reference @ cc2ec64d): the discrete-event loop `Simulator::new` + `Simulator::loop_until`
 * (bft-lib/src/simulator.rs:200-250, 380-475) driving librabft-v2's NodeState / RecordStore /
 * Pacemaker / data-sync handlers over bft-lib's SimulatedContext.  The reference has no FFI seam
 * (it is generic Rust, simulator.rs:284-295); this header is the seam a Rust shim would bind with
 * `extern "C"` (see INTEGRATION.md).  One handle runs `num_instances` independent simulator
 * instances (instance i == `Simulator::new(seeds[i], num_nodes, RandomDelay::new(mean, variance),
 * context_factory)`) in lockstep on one GPU and exposes what the reference's callers read back:
 * `committed_history()` (simulated_context.rs:98-100) and `last_committed_state()` (:194-196).
 *
 * Conventions: plain C types only; every function returns LBFT_OK (0) or a negative error code and
 * never throws or aborts across the boundary; `lbft_last_error()` gives the thread-local message.
 * A handle is not thread-safe; distinct handles are independent.  There is NO CPU fallback: if no
 * CUDA device is usable, lbft_create fails with LBFT_ERR_CUDA.
 */
#ifndef LBFT_H_
#define LBFT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LBFT_ABI_VERSION 1

enum {
  LBFT_OK = 0,
  LBFT_ERR_INVALID = -1,    /* bad argument / unsupported configuration                        */
  LBFT_ERR_CUDA = -2,       /* CUDA runtime error or no usable device                           */
  LBFT_ERR_STATE = -3,      /* call sequence error (e.g. results requested before lbft_run)     */
  LBFT_ERR_CAPACITY = -4,   /* some instance overflowed a device table; see lbft_status         */
  LBFT_ERR_NOMEM = -5
};

/* RandomDelay (simulator.rs:39-43, 99-118).  LOGNORMAL is the reference's only model.
 * UNIFORM is an extension (BASELINE.json config 2): integer uniform on [delay_lo, delay_hi]. */
enum { LBFT_DELAY_LOGNORMAL = 0, LBFT_DELAY_UNIFORM = 1 };

/* Per-instance status bits returned by lbft_status(). */
enum {
  LBFT_ST_DONE = 1u << 0,             /* event loop reached max_clock (or drained)               */
  LBFT_ST_ROUND_OVERFLOW = 1u << 1,   /* a round number reached round_cap                         */
  LBFT_ST_QUEUE_OVERFLOW = 1u << 2,   /* pending-event queue reached queue_cap                    */
  LBFT_ST_PAYLOAD_OVERFLOW = 1u << 3, /* in-flight notification pool reached payload_cap          */
  LBFT_ST_INVARIANT = 1u << 4,        /* a layout invariant (SURVEY App. C) was violated          */
  LBFT_ST_EPOCH_CHANGE = 1u << 5,     /* advisory: the instance went through an epoch change      */
                                      /* (commands_per_epoch reached, node.rs:329-348)            */
  LBFT_ST_DELAY_NEAR_INT = 1u << 6,   /* a LogNormal sample landed within 1e-9 of an integer: the */
                                      /* truncation may depend on the libm's last ulp (advisory)  */
  LBFT_ST_TIME_OVERFLOW = 1u << 7     /* a time left the 31-bit range of the device encoding      */
};
#define LBFT_ST_ERROR_MASK                                                                       \
  (LBFT_ST_ROUND_OVERFLOW | LBFT_ST_QUEUE_OVERFLOW | LBFT_ST_PAYLOAD_OVERFLOW | LBFT_ST_INVARIANT | \
   LBFT_ST_TIME_OVERFLOW)

/* One row of SimulatedContext::committed_history(): (Command{proposer,index}, NodeTime)
 * (simulated_context.rs:31-35, 98-100). */
typedef struct lbft_commit {
  uint32_t proposer;
  uint32_t index;
  int64_t time;
} lbft_commit;

/* One entry of DataWriter::nodes_round_switch (data_writer.rs:14, 34-50): at the pop of an event with
 * scheduled time `time`, node `node` was seen with ActiveRound::active_round() == `round`, larger than
 * at any earlier pop (simulator.rs:393-394: sampled after the max_clock test, before the clock max()). */
typedef struct lbft_round_switch {
  uint32_t node;
  uint32_t round;
  int64_t time;
} lbft_round_switch;

/* lbft_config.flags */
#define LBFT_FLAG_ROUND_SWITCHES 1u /* record round switches = loop_until(.., Some(csv_path)) simulator.rs:380-381 */
#define LBFT_FLAG_RESUMABLE 2u      /* lbft_run_until / snapshots: loop_until may be called again with a larger clock   */
/* NON-PARITY variant: a data-sync request is answered by the node it was SENT TO, from that node's records, and the requester
 * inserts the records of the response (what librabft-v2/src/data_sync.rs:183-240 is written for).  The reference simulator
 * dispatches the request to the requester itself (bft-lib/src/simulator.rs:446), which makes every round trip a no-op; that
 * behaviour is the default here, as its golden tests pin it.  Plain runs only (no other flag, commands_per_epoch >= round_cap). */
#define LBFT_FLAG_TRUE_DATA_SYNC 4u

/* Per-instance event counters (simulator.rs:31 event_count; data_writer.rs message counter). */
typedef struct lbft_instance_counters {
  uint32_t processed[4];      /* popped events by Event::kind(): 0 notify 1 request 2 response 3 timer */
  uint32_t timers_cancelled;  /* timer pops skipped by ignore_scheduled_updates_until (:406-410)       */
  uint32_t scheduled;         /* Simulator.event_count: creation stamps handed out                     */
  uint32_t max_active_round;  /* max over nodes of ActiveRound::active_round() (simulator.rs:86-88)     */
  uint32_t rng_draws;         /* Xoshiro256** next_u64 calls on the instance stream                    */
  uint32_t max_queue;         /* high-water mark of the device event queue (implementation-specific)   */
  uint32_t scheduled_notify;  /* DataSyncNotifyEvents handed a creation stamp (simulator.rs:348-354)    */
  uint32_t max_payloads;      /* high-water mark of in-flight notification snapshots (implementation)   */
  uint32_t timers_elided;     /* duplicate timers accounted as cancelled without being queued (impl.)  */
} lbft_instance_counters;

/* Device timing of the last lbft_run / lbft_run_device, measured with CUDA events on the stream the
 * kernels are launched on. */
typedef struct lbft_timing {
  double init_ms;        /* state-initialisation kernel                         */
  double sim_ms;         /* event-loop kernel(s)                                */
  double finalize_ms;    /* read-out kernel (commit counts + state keys)        */
  double h2d_ms, d2h_ms; /* host<->device copies inside lbft_run                */
  uint64_t h2d_bytes, d2h_bytes;
  uint32_t kernel_launches; /* kernels launched by the last run                 */
  uint32_t reserved;
} lbft_timing;

/* Batched equivalent of the arguments of `Simulator::new` + `NodeConfig` + `SimulatedContext::new`
 * + `loop_until` (simulator.rs:200-208,380; node.rs:76-81; simulated_context.rs:86; main.rs:57-172). */
typedef struct lbft_config {
  uint32_t struct_size;   /* = sizeof(lbft_config); ABI guard                                          */
  uint32_t num_instances; /* independent simulator instances                                           */
  uint32_t num_nodes;     /* main.rs --nodes (1..64)                                                   */
  uint32_t delay_kind;    /* LBFT_DELAY_*                                                              */
  const uint64_t* seeds;  /* [num_instances] host pointer; main.rs --seed, simulator.rs:212            */
  int64_t max_clock;      /* loop_until(GlobalTime(max_clock)); main.rs --max_clock                    */
  double delay_mean;      /* RandomDelay::new(mean, variance), simulator.rs:99-106                     */
  double delay_variance;
  int64_t delay_lo, delay_hi;     /* LBFT_DELAY_UNIFORM only                                           */
  int64_t target_commit_interval; /* NodeConfig, node.rs:76-81                                         */
  int64_t delta;                  /* > 0 (delta = 0 is refused: SURVEY App. C.1b)                      */
  double gamma;
  double lambda;
  uint64_t commands_per_epoch;    /* SimulatedContext::new(_, _, max_command_per_epoch)                */
  /* ---- extensions (NULL / 0 = reference behaviour; SURVEY Appendix D) ---- */
  const uint64_t* voting_rights;  /* [num_nodes] EpochConfiguration weights (configuration.rs:29-43)   */
  const uint8_t* silent;          /* [num_nodes] non-zero = silent (crashed) node                      */
  uint32_t partition_windows;     /* per-instance random partition plan: number of windows             */
  uint32_t partition_max_len;     /* maximal window length in ms                                       */
  /* ---- device / capacity tuning (0 = auto) ---- */
  int32_t device;                 /* CUDA device ordinal                                               */
  uint32_t round_cap;             /* rounds representable per instance                                 */
  uint32_t queue_cap;             /* pending events per instance                                       */
  uint32_t payload_cap;           /* in-flight notifications per instance                              */
  uint32_t flags;                 /* LBFT_FLAG_* bits; unknown bits are rejected                       */
  uint32_t reserved;
} lbft_config;

typedef struct lbft_sim lbft_sim;

/* Validate the configuration, precompute the host tables (ziggurat layers, leader per round, round
 * durations — all libm calls stay on the host), allocate device state.  Does not run anything. */
int lbft_create(const lbft_config* config, lbft_sim** out_sim);

/* One parameter set of a sweep (lbft_create_sweep): the knobs of a Monte-Carlo study — RandomDelay (simulator.rs:99-106,
 * or the uniform extension), NodeConfig (node.rs:76-81) and the silent (crashed) nodes — with lbft_config's meaning. */
typedef struct lbft_param_set {
  uint32_t struct_size;           /* = sizeof(lbft_param_set); ABI guard                                    */
  uint32_t delay_kind;            /* LBFT_DELAY_*                                                           */
  double delay_mean;
  double delay_variance;
  int64_t delay_lo, delay_hi;     /* LBFT_DELAY_UNIFORM only                                                */
  int64_t target_commit_interval;
  int64_t delta;                  /* > 0                                                                    */
  double gamma;
  double lambda;
  uint64_t silent_mask;           /* bit i set = node i is silent; bits >= num_nodes are refused            */
} lbft_param_set;

/* Largest num_sets lbft_create_sweep accepts. */
#define LBFT_MAX_PARAM_SETS 4096u

/* A sweep handle: one batch whose instances run with different parameter sets.  Instance i runs with
 * sets[set_of_instance[i]] (set_of_instance is a host array of config->num_instances entries, copied): it computes
 * exactly what instance i of an lbft_create handle computes whose config carries that set's values — same seed stream,
 * same RNG draws, same results (commit counts, state keys, commit logs, counters, status, active rounds).  The sets
 * replace config's delay_kind, delay_mean, delay_variance, delay_lo, delay_hi, target_commit_interval, delta, gamma,
 * lambda and silent: those fields of config are NOT read.  Everything else (num_nodes, max_clock, seeds,
 * commands_per_epoch, voting_rights, partition plan, capacities, device) is shared by the handle.  Each set is validated
 * like lbft_create validates a config; LBFT_ERR_INVALID also when config->flags is not 0, when commands_per_epoch <
 * round_cap (a multi-epoch layout), when num_sets is 0 or above LBFT_MAX_PARAM_SETS, or when a set index is out of
 * range.  The queue mode and capacities are chosen to fit every set.  Every other entry point works on the handle as
 * on any other (lbft_set_seeds keeps the set assignment); a sweep handle is never resumable. */
int lbft_create_sweep(const lbft_config* config, const lbft_param_set* sets, uint32_t num_sets,
                      const uint32_t* set_of_instance, lbft_sim** out_sim);

/* Simulator::new for every instance followed by loop_until(max_clock) (simulator.rs:200-250,
 * 380-475): copies the seeds host->device, runs the event-loop kernel to completion, copies the
 * per-node summaries (commit counts, last-committed-state keys, counters, status) device->host.
 * Returns LBFT_ERR_CAPACITY if any instance has a bit of LBFT_ST_ERROR_MASK set. */
int lbft_run(lbft_sim* sim);

/* Replace the seeds of the batch (a fresh `Simulator::new(seed, ..)` per instance on the next run);
 * `seeds` is a host array of num_instances entries, copied into the handle's pinned staging buffer. */
int lbft_set_seeds(lbft_sim* sim, const uint64_t* seeds);

/* The same three phases separately, for callers that keep inputs resident in HBM (bench.py `value`). */
int lbft_upload(lbft_sim* sim);     /* seeds host -> device                                  */
int lbft_run_device(lbft_sim* sim); /* init + event loop + read-out kernels, no host copies  */
int lbft_download(lbft_sim* sim);   /* summaries device -> host                              */

/* lbft_run split in two so that one host thread can drive several handles (one per GPU) at once and overlap its own
 * work with the device: lbft_run_async enqueues seeds host->device, the kernel and the summaries device->host on the
 * handle's stream and returns at once; lbft_wait blocks until they are done and reports like lbft_run
 * (lbft_run == lbft_run_async + lbft_wait).  Host staging is double-buffered: while a run is in flight the getters keep
 * serving the previous run's results, and lbft_set_seeds stages the next run's seeds without touching the buffer the
 * in-flight upload reads.  Every other entry point that touches the device returns LBFT_ERR_STATE until lbft_wait. */
int lbft_run_async(lbft_sim* sim);
int lbft_wait(lbft_sim* sim);

/* committed_history().len() per node (main.rs:47-53): out[instance * num_nodes + node]. */
int lbft_commit_counts(lbft_sim* sim, uint32_t* out);
/* last_committed_state() per node (simulated_context.rs:194-196): SipHash-1-3 key of the log. */
int lbft_last_states(lbft_sim* sim, uint64_t* out);
/* committed_history() of one node; writes min(*n, cap) rows, *n = full length. */
int lbft_commit_log(lbft_sim* sim, uint32_t instance, uint32_t node, lbft_commit* out, size_t cap, size_t* n);
/* committed_history() of EVERY context of the batch in one device pass and one copy (simulated_context.rs:98-100):
 * out[instance * cap + k], k < cap, is row k of the instance's longest log, and every node's committed_history() is
 * its first lens[instance * num_nodes + node] rows — the logs of one instance are prefixes of one chain because a
 * commit extends the previous one by exactly one block (simulated_context.rs:172-174); the device verifies it and
 * the call fails with LBFT_ERR_STATE if it does not hold for some instance (then read that instance with
 * lbft_commit_log).  Rows past a log's end are zero; logs longer than cap are truncated (lens tells).  lens may be
 * NULL. */
int lbft_commit_logs(lbft_sim* sim, lbft_commit* out, size_t cap, uint32_t* lens);
/* Round switches of one instance (needs LBFT_FLAG_ROUND_SWITCHES, else LBFT_ERR_STATE): node-major,
 * rounds ascending within a node; writes min(*n, cap) rows, *n = full length.  Replaces the data behind
 * DataWriter::write_to_file's round_switches.txt (data_writer.rs:61-86); number_of_messages.txt is
 * processed[0] + processed[1] + processed[2] of lbft_counters. */
int lbft_round_switches(lbft_sim* sim, uint32_t instance, lbft_round_switch* out, size_t cap, size_t* n);
/* max over nodes of ActiveRound::active_round() per instance (simulator.rs:86-88): out[num_instances].  The same
 * number as lbft_instance_counters.max_active_round, without copying the whole counter table — it is the unit of
 * the throughput metric (simulated consensus rounds). */
int lbft_active_rounds(lbft_sim* sim, uint32_t* out);
/* Per-instance counters and status flags: out[num_instances]. */
int lbft_counters(lbft_sim* sim, lbft_instance_counters* out);
int lbft_status(lbft_sim* sim, uint32_t* out);
int lbft_timing_info(lbft_sim* sim, lbft_timing* out);
/* Name of the kernel instantiation this handle launches, spelled like the symbol ncu and cuobjdump show (the host picks
 * it from the configuration: committee size, horizon, capacities, flags); NUL-terminated, truncated to cap. */
int lbft_kernel_info(lbft_sim* sim, char* buf, size_t cap);
/* Bytes of device memory held by the handle, and the per-instance state footprint. */
int lbft_memory_info(lbft_sim* sim, uint64_t* device_bytes, uint32_t* words_per_instance);

/* Resumable runs (needs LBFT_FLAG_RESUMABLE, else LBFT_ERR_STATE).  lbft_config.max_clock is the FINAL horizon the
 * device tables are sized for; lbft_run_until(sim, t), 0 <= t <= max_clock, is loop_until(GlobalTime(t), ..)
 * (simulator.rs:380-475) on every instance: the first call is Simulator::new + loop_until, each later call continues
 * where the previous one stopped — including the reference's own exit behaviour: the first event beyond t is popped
 * and dropped (simulator.rs:383-391), so a staged run is NOT the same simulation as a one-shot run to the same
 * clock.  Results (all getters) describe the state at the stop.  lbft_run / lbft_upload / lbft_set_seeds start over. */
int lbft_run_until(lbft_sim* sim, int64_t stop_clock);
/* Checkpoint of the whole batch between two lbft_run_until calls (the batched analogue of
 * ConsensusNode::save_node / load_node, librabft-v2/src/node.rs:211-238, plus the simulator's own queue, clock and
 * RNG): save after a lbft_run_until, load into a handle created from the same configuration (verified by a digest;
 * LBFT_ERR_INVALID otherwise), then continue with lbft_run_until. */
int lbft_snapshot_size(lbft_sim* sim, size_t* bytes);
int lbft_snapshot_save(lbft_sim* sim, void* buf, size_t cap);
int lbft_snapshot_load(lbft_sim* sim, const void* buf, size_t bytes);

/* Device address of a result buffer, for callers that consume results on the GPU (e.g. an NCCL
 * all-gather of per-instance commit counts): which = 0 commit counts [I][N] u32, 1 last states [I][N]
 * u64, 2 counters [I][12] u32, 3 status [I] u32, 4 active rounds [I] u32, 5 = buffers 1, 0 and 4 as the one contiguous block they are
 * allocated in (last states, commit counts, active rounds — in this order): the summaries of a shard in a single collective.
 * Valid until lbft_destroy. */
int lbft_device_buffer(lbft_sim* sim, uint32_t which, void** device_ptr, size_t* bytes);

void lbft_destroy(lbft_sim* sim);
const char* lbft_last_error(void);
uint32_t lbft_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* LBFT_H_ */
