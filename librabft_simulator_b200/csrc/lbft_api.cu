// lbft_api.cu — the C ABI of include/lbft.h over the sm_100a event-loop kernel.
//
// Replaces, for a whole batch of instances at once, the reference call sequence
//   Simulator::new(seed, nodes, RandomDelay::new(mean, variance), context_factory)   simulator.rs:200-250
//   sim.loop_until(GlobalTime(max_clock), None)                                      simulator.rs:380-475
//   contexts[i].committed_history() / last_committed_state()                         simulated_context.rs:98-100,194-196
// (callers: librabft-v2/src/main.rs:36-53, librabft-v2/tests/simulated_run.rs:19-94).
// There is no CPU fallback: without a usable CUDA device every entry point fails with LBFT_ERR_CUDA.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/lbft.h"
#include "host_setup.hpp"
#include "kernels.cuh"

using namespace lbft;

#define LBFT_SAME(a, b) ((uint32_t)(a) == (uint32_t)(b))
static_assert(LBFT_SAME(ST_DONE, LBFT_ST_DONE) && LBFT_SAME(ST_ROUND_OVERFLOW, LBFT_ST_ROUND_OVERFLOW) &&
                  LBFT_SAME(ST_QUEUE_OVERFLOW, LBFT_ST_QUEUE_OVERFLOW) && LBFT_SAME(ST_PAYLOAD_OVERFLOW, LBFT_ST_PAYLOAD_OVERFLOW) &&
                  LBFT_SAME(ST_INVARIANT, LBFT_ST_INVARIANT) && LBFT_SAME(ST_EPOCH_CHANGE, LBFT_ST_EPOCH_CHANGE) &&
                  LBFT_SAME(ST_DELAY_NEAR_INT, LBFT_ST_DELAY_NEAR_INT) && LBFT_SAME(ST_TIME_OVERFLOW, LBFT_ST_TIME_OVERFLOW),
              "status bits out of sync with include/lbft.h");
static_assert(sizeof(lbft_instance_counters) == 12 * sizeof(uint32_t), "counter layout");
static_assert(LBFT_SAME(ST_ERROR_BITS, LBFT_ST_ERROR_MASK), "error mask out of sync with include/lbft.h");

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
static int set_error(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                                   \
  do {                                                                                                   \
    cudaError_t e_ = (expr);                                                                             \
    if (e_ != cudaSuccess)                                                                               \
      return set_error(LBFT_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));             \
  } while (0)

// Pinned host mirrors of one run's summaries.  There are two sets: an asynchronous run fills the one the getters are not
// reading, so the results of run k stay readable while run k+1 is in flight (lbft_run_async / lbft_wait).
struct HostResults {
  uint32_t* commit_counts = nullptr;
  uint32_t* lc_round = nullptr;
  uint64_t* last_state = nullptr;
  uint32_t* counters = nullptr;
  uint32_t* status = nullptr;
  uint32_t* rounds = nullptr;
  uint32_t* error = nullptr;  // [1] OR of the status words with an error bit
};

struct lbft_sim {
  HostSetup hs;
  Params P{};
  int device = 0;
  uint32_t I = 0, N = 0;
  uint32_t stride = 32;  // instances per tile (the lane-interleaving factor of the state layout)
  std::vector<uint64_t> seeds_host;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[6] = {};
  // device buffers
  uint64_t* d_seeds = nullptr;
  double* d_zx = nullptr;
  double* d_zf = nullptr;
  uint8_t* d_leader = nullptr;
  int32_t* d_duration = nullptr;
  int32_t* d_period = nullptr;
  uint32_t* d_weights = nullptr;
  double* d_delay_thr = nullptr;
  // sweep handles (lbft_create_sweep): the per-set tables and each instance's set
  SweepSet* d_sets = nullptr;
  uint32_t* d_set_of = nullptr;
  double* d_sweep_thr = nullptr;
  int32_t* d_sweep_duration = nullptr;
  int32_t* d_sweep_period = nullptr;
  uint32_t* d_state = nullptr;
  uint32_t* d_commit_counts = nullptr;
  uint32_t* d_lc_round = nullptr;
  uint64_t* d_last_state = nullptr;
  uint32_t* d_counters = nullptr;
  uint32_t* d_status = nullptr;
  uint32_t* d_rounds = nullptr;
  uint32_t* d_error = nullptr;
  // d_last_state, d_commit_counts and d_rounds are carved out of ONE allocation, in this order, so that the per-instance
  // summaries a multi-GPU caller all-gathers travel in a single collective (lbft_device_buffer(5))
  unsigned char* d_summary = nullptr;
  size_t summary_bytes = 0;
  lbft_commit* d_logs = nullptr;  // lbft_commit_logs: [I][logs_cap], allocated on first use
  size_t logs_cap = 0;
  uint64_t device_bytes = 0;
  // pinned host staging: two seed buffers (lbft_set_seeds never writes the one an in-flight upload reads) and two
  // result sets (see HostResults)
  uint64_t* h_seeds[2] = {nullptr, nullptr};
  int seed_set = 0;        // buffer holding the most recently set seeds
  int seed_inflight = -1;  // buffer an in-flight upload is reading, -1 if none
  HostResults res[2];
  int done = 0;            // result set the getters read
  bool pending = false;    // an lbft_run_async has not been waited for
  bool pending_download = false;  // ... and it includes the device->host copies
  bool uploaded = false, ran = false, downloaded = false;
  bool started = false;     // resumable handles: a staged run is in progress, the next launch restores the instances
  int64_t next_stop = 0;    // stop clock of the next launch (max_clock unless set by lbft_run_until)
  int64_t last_stop = -1;   // stop clock of the last launch
  lbft_timing timing{};
};

template <class T>
static cudaError_t dev_alloc(lbft_sim* s, T** p, size_t count) {
  cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
  if (e == cudaSuccess) s->device_bytes += count * sizeof(T);
  return e;
}

static void free_all(lbft_sim* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);  // an lbft_run_async may still be in flight
  cudaFree(s->d_seeds); cudaFree(s->d_zx); cudaFree(s->d_zf); cudaFree(s->d_leader); cudaFree(s->d_duration);
  cudaFree(s->d_period); cudaFree(s->d_weights); cudaFree(s->d_delay_thr); cudaFree(s->d_state); cudaFree(s->d_summary);
  cudaFree(s->d_lc_round); cudaFree(s->d_counters); cudaFree(s->d_status);
  cudaFree(s->d_error); cudaFree(s->d_logs);
  cudaFree(s->d_sets); cudaFree(s->d_set_of); cudaFree(s->d_sweep_thr); cudaFree(s->d_sweep_duration); cudaFree(s->d_sweep_period);
  for (int b = 0; b < 2; b++) {
    cudaFreeHost(s->h_seeds[b]);
    HostResults& r = s->res[b];
    cudaFreeHost(r.commit_counts); cudaFreeHost(r.lc_round); cudaFreeHost(r.last_state); cudaFreeHost(r.counters);
    cudaFreeHost(r.status); cudaFreeHost(r.rounds); cudaFreeHost(r.error);
  }
  for (auto& e : s->ev)
    if (e) cudaEventDestroy(e);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

// The three phases of a run, enqueued on the handle's stream without waiting.
static int enqueue_upload(lbft_sim* s) {
  CUDA_TRY(cudaEventRecord(s->ev[0], s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->d_seeds, s->h_seeds[s->seed_set], s->I * sizeof(uint64_t), cudaMemcpyHostToDevice, s->stream));
  CUDA_TRY(cudaEventRecord(s->ev[1], s->stream));
  s->seed_inflight = s->seed_set;
  return LBFT_OK;
}
static int enqueue_kernel(lbft_sim* s);
static int enqueue_download(lbft_sim* s, HostResults& r) {
  const size_t I = s->I, N = s->N;
  CUDA_TRY(cudaEventRecord(s->ev[4], s->stream));
  CUDA_TRY(cudaMemcpyAsync(r.commit_counts, s->d_commit_counts, I * N * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(r.lc_round, s->d_lc_round, I * N * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(r.last_state, s->d_last_state, I * N * sizeof(uint64_t), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(r.counters, s->d_counters, I * 12 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(r.status, s->d_status, I * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(r.rounds, s->d_rounds, I * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(r.error, s->d_error, sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaEventRecord(s->ev[5], s->stream));
  return LBFT_OK;
}
// After the stream has drained: timings, and the one-word error check (the per-instance statuses are only scanned
// to name the first offender when the device-side OR says there is one).
static int finish_upload(lbft_sim* s) {
  float ms = 0;
  CUDA_TRY(cudaEventElapsedTime(&ms, s->ev[0], s->ev[1]));
  s->timing.h2d_ms = ms;
  s->timing.h2d_bytes = s->I * sizeof(uint64_t);
  s->seed_inflight = -1;
  s->uploaded = true;
  return LBFT_OK;
}
static int finish_kernel(lbft_sim* s) {
  float ms = 0;
  CUDA_TRY(cudaEventElapsedTime(&ms, s->ev[2], s->ev[3]));
  s->timing.init_ms = 0;
  s->timing.sim_ms = ms;
  s->timing.finalize_ms = 0;
  s->timing.kernel_launches = 1;
  s->ran = true;
  s->downloaded = false;
  s->started = s->P.resumable != 0;
  s->last_stop = s->P.stop_clock;
  return LBFT_OK;
}
static int finish_download(lbft_sim* s, int set) {
  float ms = 0;
  CUDA_TRY(cudaEventElapsedTime(&ms, s->ev[4], s->ev[5]));
  const size_t I = s->I, N = s->N;
  s->timing.d2h_ms = ms;
  s->timing.d2h_bytes = I * N * (2 * sizeof(uint32_t) + sizeof(uint64_t)) + I * 14 * sizeof(uint32_t) + sizeof(uint32_t);
  s->done = set;
  s->downloaded = true;
  const HostResults& r = s->res[set];
  if (*r.error & LBFT_ST_ERROR_MASK) {
    for (size_t i = 0; i < I; i++)
      if (r.status[i] & LBFT_ST_ERROR_MASK) {
        char buf[360];
        snprintf(buf, sizeof buf, "instance %zu ended with status 0x%x (see lbft_status; raise round_cap/queue_cap/payload_cap%s)", i,
                 r.status[i], (r.status[i] & LBFT_ST_QUEUE_OVERFLOW) ? "; QUEUE_OVERFLOW also means the queue mode ran out of creation "
                 "stamps: queue_cap > 512 selects a queue with wider stamps" : "");
        return set_error(LBFT_ERR_CAPACITY, buf);
      }
  }
  return LBFT_OK;
}
static int need_idle(lbft_sim* s) {
  if (!s) return set_error(LBFT_ERR_INVALID, "sim must not be NULL");
  if (s->pending) return set_error(LBFT_ERR_STATE, "an lbft_run_async is in flight: call lbft_wait first");
  return LBFT_OK;
}

static int create_handle(lbft_sim* s, const lbft_config* config, lbft_sim** out_sim);

extern "C" {

uint32_t lbft_abi_version(void) { return LBFT_ABI_VERSION; }
const char* lbft_last_error(void) { return g_last_error.c_str(); }

int lbft_create(const lbft_config* config, lbft_sim** out_sim) {
  if (!config || !out_sim) return set_error(LBFT_ERR_INVALID, "config and out_sim must not be NULL");
  *out_sim = nullptr;
  lbft_sim* s = new (std::nothrow) lbft_sim();
  if (!s) return set_error(LBFT_ERR_NOMEM, "out of host memory");
  if (!s->hs.build(*config)) {
    std::string e = s->hs.error;
    delete s;
    return set_error(LBFT_ERR_INVALID, e);
  }
  if (s->hs.params.L.epochs > 1 && (s->hs.params.record_rs || s->hs.params.resumable)) {
    delete s;
    return set_error(LBFT_ERR_INVALID, "recording / resumable handles need commands_per_epoch >= round_cap: the kernels with the epoch "
                                       "machinery (node.rs:329-348) are built for plain runs only");
  }
  return create_handle(s, config, out_sim);
}

int lbft_create_sweep(const lbft_config* config, const lbft_param_set* sets, uint32_t num_sets, const uint32_t* set_of_instance,
                      lbft_sim** out_sim) {
  if (!config || !out_sim) return set_error(LBFT_ERR_INVALID, "config and out_sim must not be NULL");
  *out_sim = nullptr;
  lbft_sim* s = new (std::nothrow) lbft_sim();
  if (!s) return set_error(LBFT_ERR_NOMEM, "out of host memory");
  if (!s->hs.build_sweep(*config, sets, num_sets, set_of_instance)) {
    std::string e = s->hs.error;
    delete s;
    return set_error(LBFT_ERR_INVALID, e);
  }
  return create_handle(s, config, out_sim);
}

}  // extern "C"

// The device side of lbft_create / lbft_create_sweep once the host setup has been built and validated.
static int create_handle(lbft_sim* s, const lbft_config* config, lbft_sim** out_sim) {
  s->I = config->num_instances;
  s->N = config->num_nodes;
  s->device = config->device;
  s->stride = s->hs.tile_stride;
  s->seeds_host.assign(config->seeds, config->seeds + s->I);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    delete s;
    return set_error(LBFT_ERR_CUDA, std::string("no usable CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
  }
  if (s->device < 0 || s->device >= ndev) {
    delete s;
    return set_error(LBFT_ERR_INVALID, "device ordinal out of range");
  }
#define CREATE_TRY(expr)                                                                      \
  do {                                                                                        \
    cudaError_t e2_ = (expr);                                                                 \
    if (e2_ != cudaSuccess) {                                                                 \
      std::string m_ = std::string(#expr) + ": " + cudaGetErrorString(e2_);                 \
      free_all(s);                                                                            \
      return set_error(e2_ == cudaErrorMemoryAllocation ? LBFT_ERR_NOMEM : LBFT_ERR_CUDA, m_); \
    }                                                                                         \
  } while (0)
  CREATE_TRY(cudaSetDevice(s->device));
  CREATE_TRY(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
  for (auto& evt : s->ev) CREATE_TRY(cudaEventCreate(&evt));
  const Layout& L = s->hs.params.L;
  const size_t I = s->I, N = s->N, tiles = (I + s->stride - 1) / s->stride;
  CREATE_TRY(dev_alloc(s, &s->d_seeds, I));
  CREATE_TRY(dev_alloc(s, &s->d_zx, 257));
  CREATE_TRY(dev_alloc(s, &s->d_zf, 257));
  CREATE_TRY(dev_alloc(s, &s->d_leader, s->hs.leader.size()));
  CREATE_TRY(dev_alloc(s, &s->d_duration, s->hs.duration.size()));
  CREATE_TRY(dev_alloc(s, &s->d_period, s->hs.period.size()));
  CREATE_TRY(dev_alloc(s, &s->d_weights, N));
  if (!s->hs.delay_thr.empty()) CREATE_TRY(dev_alloc(s, &s->d_delay_thr, s->hs.delay_thr.size()));
  CREATE_TRY(dev_alloc(s, &s->d_state, tiles * L.total_words * s->stride));
  s->summary_bytes = I * N * sizeof(uint64_t) + I * N * sizeof(uint32_t) + I * sizeof(uint32_t);
  CREATE_TRY(dev_alloc(s, &s->d_summary, s->summary_bytes));
  s->d_last_state = reinterpret_cast<uint64_t*>(s->d_summary);
  s->d_commit_counts = reinterpret_cast<uint32_t*>(s->d_summary + I * N * sizeof(uint64_t));
  s->d_rounds = s->d_commit_counts + I * N;
  CREATE_TRY(dev_alloc(s, &s->d_lc_round, I * N));
  CREATE_TRY(dev_alloc(s, &s->d_counters, I * 12));
  CREATE_TRY(dev_alloc(s, &s->d_status, I));
  CREATE_TRY(dev_alloc(s, &s->d_error, 1));
  for (int b = 0; b < 2; b++) {
    HostResults& r = s->res[b];
    CREATE_TRY(cudaMallocHost((void**)&s->h_seeds[b], I * sizeof(uint64_t)));
    CREATE_TRY(cudaMallocHost((void**)&r.commit_counts, I * N * sizeof(uint32_t)));
    CREATE_TRY(cudaMallocHost((void**)&r.lc_round, I * N * sizeof(uint32_t)));
    CREATE_TRY(cudaMallocHost((void**)&r.last_state, I * N * sizeof(uint64_t)));
    CREATE_TRY(cudaMallocHost((void**)&r.counters, I * 12 * sizeof(uint32_t)));
    CREATE_TRY(cudaMallocHost((void**)&r.status, I * sizeof(uint32_t)));
    CREATE_TRY(cudaMallocHost((void**)&r.rounds, I * sizeof(uint32_t)));
    CREATE_TRY(cudaMallocHost((void**)&r.error, sizeof(uint32_t)));
  }
  memcpy(s->h_seeds[0], s->seeds_host.data(), I * sizeof(uint64_t));
  // launch-invariant tables
  CREATE_TRY(cudaMemcpy(s->d_zx, s->hs.zig_x.data(), 257 * sizeof(double), cudaMemcpyHostToDevice));
  CREATE_TRY(cudaMemcpy(s->d_zf, s->hs.zig_f.data(), 257 * sizeof(double), cudaMemcpyHostToDevice));
  CREATE_TRY(cudaMemcpy(s->d_leader, s->hs.leader.data(), s->hs.leader.size(), cudaMemcpyHostToDevice));
  CREATE_TRY(cudaMemcpy(s->d_duration, s->hs.duration.data(), s->hs.duration.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  CREATE_TRY(cudaMemcpy(s->d_period, s->hs.period.data(), s->hs.period.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  CREATE_TRY(cudaMemcpy(s->d_weights, s->hs.weights.data(), N * sizeof(uint32_t), cudaMemcpyHostToDevice));
  if (s->d_delay_thr)
    CREATE_TRY(cudaMemcpy(s->d_delay_thr, s->hs.delay_thr.data(), s->hs.delay_thr.size() * sizeof(double), cudaMemcpyHostToDevice));
  const HostSetup& hs = s->hs;
  if (!hs.sets.empty()) {
    CREATE_TRY(dev_alloc(s, &s->d_sets, hs.sets.size()));
    CREATE_TRY(dev_alloc(s, &s->d_set_of, I));
    CREATE_TRY(dev_alloc(s, &s->d_sweep_duration, hs.sweep_duration.size()));
    CREATE_TRY(dev_alloc(s, &s->d_sweep_period, hs.sweep_period.size()));
    if (!hs.sweep_thr.empty()) CREATE_TRY(dev_alloc(s, &s->d_sweep_thr, hs.sweep_thr.size()));
    CREATE_TRY(cudaMemcpy(s->d_sets, hs.sets.data(), hs.sets.size() * sizeof(SweepSet), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(s->d_set_of, hs.set_of.data(), I * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(s->d_sweep_duration, hs.sweep_duration.data(), hs.sweep_duration.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(s->d_sweep_period, hs.sweep_period.data(), hs.sweep_period.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    if (s->d_sweep_thr)
      CREATE_TRY(cudaMemcpy(s->d_sweep_thr, hs.sweep_thr.data(), hs.sweep_thr.size() * sizeof(double), cudaMemcpyHostToDevice));
  }
#undef CREATE_TRY
  s->P = s->hs.params;
  s->P.seeds = s->d_seeds;
  s->P.zig_x = s->d_zx;
  s->P.zig_f = s->d_zf;
  s->P.leader = s->d_leader;
  s->P.duration = s->d_duration;
  s->P.period = s->d_period;
  s->P.weights = s->d_weights;
  s->P.delay_thr = s->d_delay_thr;
  s->P.state = s->d_state;
  s->P.out_commit_counts = s->d_commit_counts;
  s->P.out_lc_round = s->d_lc_round;
  s->P.out_last_state = s->d_last_state;
  s->P.out_counters = s->d_counters;
  s->P.out_status = s->d_status;
  s->P.out_rounds = s->d_rounds;
  s->P.out_error = s->d_error;
  s->P.sweep_sets = s->d_sets;
  s->P.set_of = s->d_set_of;
  s->P.sweep_thr = s->d_sweep_thr;
  s->P.sweep_duration = s->d_sweep_duration;
  s->P.sweep_period = s->d_sweep_period;
  s->P.num_sets = (uint32_t)hs.sets.size();
  *out_sim = s;
  return LBFT_OK;
}

extern "C" {

int lbft_set_seeds(lbft_sim* s, const uint64_t* seeds) {
  if (!s || !seeds) return set_error(LBFT_ERR_INVALID, "NULL argument");
  // never the buffer an in-flight upload is reading (lbft_run_async): the caller may stage run k+1 while run k runs
  const int b = s->seed_set != s->seed_inflight ? s->seed_set : 1 - s->seed_set;
  memcpy(s->h_seeds[b], seeds, (size_t)s->I * sizeof(uint64_t));
  s->seed_set = b;
  s->uploaded = false;
  s->started = false;
  return LBFT_OK;
}

int lbft_device_buffer(lbft_sim* s, uint32_t which, void** device_ptr, size_t* bytes) {
  if (!s || !device_ptr || !bytes) return set_error(LBFT_ERR_INVALID, "NULL argument");
  const size_t I = s->I, N = s->N;
  switch (which) {
    case 0: *device_ptr = s->d_commit_counts; *bytes = I * N * sizeof(uint32_t); break;
    case 1: *device_ptr = s->d_last_state; *bytes = I * N * sizeof(uint64_t); break;
    case 2: *device_ptr = s->d_counters; *bytes = I * 12 * sizeof(uint32_t); break;
    case 3: *device_ptr = s->d_status; *bytes = I * sizeof(uint32_t); break;
    case 4: *device_ptr = s->d_rounds; *bytes = I * sizeof(uint32_t); break;
    case 5: *device_ptr = s->d_summary; *bytes = s->summary_bytes; break;
    default: return set_error(LBFT_ERR_INVALID, "unknown buffer id");
  }
  return LBFT_OK;
}

int lbft_upload(lbft_sim* s) {
  if (int r = need_idle(s)) return r;
  CUDA_TRY(cudaSetDevice(s->device));
  if (int r = enqueue_upload(s)) return r;
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (int r = finish_upload(s)) return r;
  s->started = false;  // fresh seeds: the next launch is Simulator::new
  s->next_stop = s->P.max_clock;
  return LBFT_OK;
}

int lbft_run_device(lbft_sim* s) {
  if (int r = need_idle(s)) return r;
  if (!s->uploaded) return set_error(LBFT_ERR_STATE, "lbft_upload must be called before lbft_run_device");
  CUDA_TRY(cudaSetDevice(s->device));
  if (int r = enqueue_kernel(s)) return r;
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return finish_kernel(s);
}

int lbft_download(lbft_sim* s) {
  if (int r = need_idle(s)) return r;
  if (!s->ran) return set_error(LBFT_ERR_STATE, "nothing has been run yet");
  CUDA_TRY(cudaSetDevice(s->device));
  const int set = 1 - s->done;
  if (int r = enqueue_download(s, s->res[set])) return r;
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return finish_download(s, set);
}

// lbft_run = lbft_run_async + lbft_wait.
int lbft_run_async(lbft_sim* s) {
  if (int r = need_idle(s)) return r;
  CUDA_TRY(cudaSetDevice(s->device));
  s->next_stop = s->P.max_clock;
  s->started = false;
  if (int r = enqueue_upload(s)) return r;
  s->uploaded = true;
  if (int r = enqueue_kernel(s)) return r;
  if (int r = enqueue_download(s, s->res[1 - s->done])) return r;
  s->pending = true;
  return LBFT_OK;
}

int lbft_wait(lbft_sim* s) {
  if (!s) return set_error(LBFT_ERR_INVALID, "sim must not be NULL");
  if (!s->pending) return set_error(LBFT_ERR_STATE, "no lbft_run_async is in flight");
  CUDA_TRY(cudaSetDevice(s->device));
  s->pending = false;
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (int r = finish_upload(s)) return r;
  if (int r = finish_kernel(s)) return r;
  return finish_download(s, 1 - s->done);
}

int lbft_run(lbft_sim* s) {
  if (int r = lbft_run_async(s)) return r;
  return lbft_wait(s);
}

int lbft_run_until(lbft_sim* s, int64_t stop_clock) {
  if (int r = need_idle(s)) return r;
  if (!s->P.resumable) return set_error(LBFT_ERR_STATE, "not a resumable handle: set LBFT_FLAG_RESUMABLE in lbft_config.flags");
  if (stop_clock < 0 || stop_clock > s->P.max_clock)
    return set_error(LBFT_ERR_INVALID, "stop_clock must be in [0, lbft_config.max_clock] (the horizon the device tables are sized for)");
  if (!s->started) {
    int r = lbft_upload(s);  // Simulator::new on the next launch
    if (r != LBFT_OK) return r;
  }
  s->next_stop = stop_clock;
  int r = lbft_run_device(s);
  if (r != LBFT_OK) return r;
  return lbft_download(s);
}

}  // extern "C"

// Which instantiation this handle launches (host_setup.hpp decided wide vs thread-per-instance and the queue mode).
static KernelSel select_kernel(const lbft_sim* s) {
  KernelSel k{};
  k.wide = s->hs.use_wide;
  k.smem = s->hs.wide_smem;
  k.group = (int)s->hs.wide_group;
  k.epochs = s->P.L.epochs > 1;
  k.tds = s->P.L.tds != 0;
  k.tile = (int)s->stride;
  k.qmode = (int)s->P.L.queue_scan;
  k.nmax = (k.qmode == 1 || k.qmode == 2) ? 16 : (s->N <= 16 ? 16 : (s->N <= 32 ? 32 : 64));
  k.rec = s->P.record_rs != 0;
  k.res = s->P.resumable != 0;
  k.sweep = s->P.num_sets != 0;
  // shapes with a kernel instantiation with compile-time field offsets (sim_params.h fixed_layout): the handle's layout must
  // be bit-identical and the delay model the reference's (LogNormal served by the threshold table)
  constexpr Layout kDefault4 = fixed_layout(FX_DEFAULT4), kPart7 = fixed_layout(FX_PART7), kCommittee64 = fixed_layout(FX_COMMITTEE64);
  const bool table_delay = s->P.delay_kind == LBFT_DELAY_LOGNORMAL && !s->P.delay_const && s->P.delay_kmax != 0;
  const bool plain_model = table_delay && s->P.delay_kmax + 2 <= kThrSmem && s->P.silent_mask == 0;
  const bool plain_handle = !k.rec && !k.res && !k.tds && !k.epochs;
  k.fixed = FX_NONE;
  if (k.sweep) return k;  // (the sweep kernels have no compile-time layouts)
  if (!k.wide && k.qmode == 2 && plain_model && plain_handle && memcmp(&s->P.L, &kDefault4, sizeof(Layout)) == 0) k.fixed = FX_DEFAULT4;
  else if (!k.wide && k.qmode == 3 && k.tile == 8 && plain_model && plain_handle && memcmp(&s->P.L, &kPart7, sizeof(Layout)) == 0) k.fixed = FX_PART7;
  else if (k.wide && k.qmode == 3 && k.group == 8 && !k.smem && table_delay && plain_handle && memcmp(&s->P.L, &kCommittee64, sizeof(Layout)) == 0)
    k.fixed = FX_COMMITTEE64;
  if (const char* f = std::getenv("LBFT_NO_FIXED_SHAPES"))  // A/B runs: the generic instantiations for the shapes other than the default one
    if (atoi(f) != 0 && k.fixed != FX_DEFAULT4) k.fixed = FX_NONE;
  return k;
}
// ... spelled like the symbol ncu / cuobjdump show.
static std::string kernel_name(const lbft_sim* s) {
  const KernelSel k = select_kernel(s);
  char buf[96];
  if (k.sweep && k.wide)
    snprintf(buf, sizeof buf, "lbft_sweep_wide_kernel<%d,%d,%s,%d>", k.nmax, k.qmode, k.smem ? "true" : "false", k.group);
  else if (k.sweep)
    snprintf(buf, sizeof buf, "lbft_sweep_kernel<%d,%d>", k.nmax, k.qmode);
  else if (k.wide)
    snprintf(buf, sizeof buf, "lbft_wide_kernel<%d,%d,%s,%d,%s,%d>", k.nmax, k.qmode, k.smem ? "true" : "false", k.group, k.epochs ? "true" : "false", k.fixed);
  else
    snprintf(buf, sizeof buf, "lbft_event_loop_kernel<%d,%d,%d,%s,%s,%s,%s,%d>", k.nmax, k.qmode, k.fixed, k.rec ? "true" : "false",
             k.res ? "true" : "false", k.epochs ? "true" : "false", k.tds ? "true" : "false", k.tile);
  return buf;
}

static int enqueue_kernel(lbft_sim* s) {
  s->P.stop_clock = (int32_t)(s->P.resumable ? s->next_stop : (int64_t)s->P.max_clock);
  s->P.run_flags = (s->P.resumable && s->started) ? 1u : 0u;
  CUDA_TRY(cudaMemsetAsync(s->d_error, 0, sizeof(uint32_t), s->stream));
  CUDA_TRY(cudaEventRecord(s->ev[2], s->stream));
  const KernelSel k = select_kernel(s);
  cudaError_t e = k.sweep ? (k.wide ? launch_sweep_wide(k, s->P, s->stream) : launch_sweep(k, s->P, s->stream))
                  : k.wide ? launch_wide(k, s->P, s->stream)
                  : k.fixed == FX_DEFAULT4 ? launch_fixed(k, s->P, s->stream)
                  : (k.qmode == 1 || k.qmode == 2) ? launch_scan(k, s->P, s->stream)
                  : k.qmode == 3 ? launch_calendar(k, s->P, s->stream)
                                 : launch_heap(k, s->P, s->stream);
  if (e != cudaSuccess) return set_error(LBFT_ERR_CUDA, std::string("kernel launch (") + kernel_name(s) + "): " + cudaGetErrorString(e));
  CUDA_TRY(cudaEventRecord(s->ev[3], s->stream));
  return LBFT_OK;
}

extern "C" {

// ---- snapshots: header + the state tiles (which hold the save areas of a resumable handle) ----
namespace {
struct SnapshotHeader {
  uint64_t magic;  // "LBFTSNP1"
  uint32_t abi, num_instances, num_nodes, total_words;
  int64_t max_clock, last_stop;
  uint64_t config_digest;
};
constexpr uint64_t kSnapMagic = 0x31504e535446424cULL;
uint64_t fnv1a(uint64_t h, const void* p, size_t n) {
  const unsigned char* b = static_cast<const unsigned char*>(p);
  for (size_t i = 0; i < n; i++) { h ^= b[i]; h *= 0x100000001b3ULL; }
  return h;
}
// Everything that shapes the simulation except the seeds: the scalar part of Params (layout, delay model, quorum,
// voting rights, ...) and the host tables.
uint64_t config_digest(const lbft_sim* s) {
  Params q = s->P;
  q.stop_clock = 0; q.run_flags = 0;
  uint64_t h = fnv1a(0xcbf29ce484222325ULL, &q, offsetof(Params, seeds));
  h = fnv1a(h, s->hs.leader.data(), s->hs.leader.size());
  h = fnv1a(h, s->hs.duration.data(), s->hs.duration.size() * sizeof(int32_t));
  h = fnv1a(h, s->hs.period.data(), s->hs.period.size() * sizeof(int32_t));
  if (!s->hs.delay_thr.empty()) h = fnv1a(h, s->hs.delay_thr.data(), s->hs.delay_thr.size() * sizeof(double));
  return h;
}
size_t state_bytes(const lbft_sim* s) { return (size_t)((s->I + s->stride - 1) / s->stride) * s->P.L.total_words * s->stride * sizeof(uint32_t); }
}  // namespace

int lbft_snapshot_size(lbft_sim* s, size_t* bytes) {
  if (!s || !bytes) return set_error(LBFT_ERR_INVALID, "NULL argument");
  if (!s->P.resumable) return set_error(LBFT_ERR_STATE, "not a resumable handle: set LBFT_FLAG_RESUMABLE in lbft_config.flags");
  *bytes = sizeof(SnapshotHeader) + state_bytes(s);
  return LBFT_OK;
}

int lbft_snapshot_save(lbft_sim* s, void* buf, size_t cap) {
  size_t need = 0;
  if (int r = lbft_snapshot_size(s, &need)) return r;
  if (!buf || cap < need) return set_error(LBFT_ERR_INVALID, "snapshot buffer too small (see lbft_snapshot_size)");
  if (!s->started) return set_error(LBFT_ERR_STATE, "nothing to snapshot: call lbft_run_until first");
  if (int r = need_idle(s)) return r;
  CUDA_TRY(cudaSetDevice(s->device));
  SnapshotHeader h{kSnapMagic, LBFT_ABI_VERSION, s->I, s->N, s->P.L.total_words, s->P.max_clock, s->last_stop, config_digest(s)};
  memcpy(buf, &h, sizeof h);
  CUDA_TRY(cudaMemcpy(static_cast<char*>(buf) + sizeof h, s->d_state, state_bytes(s), cudaMemcpyDeviceToHost));
  return LBFT_OK;
}

int lbft_snapshot_load(lbft_sim* s, const void* buf, size_t bytes) {
  size_t need = 0;
  if (int r = lbft_snapshot_size(s, &need)) return r;
  if (!buf || bytes < sizeof(SnapshotHeader)) return set_error(LBFT_ERR_INVALID, "not a snapshot");
  SnapshotHeader h;
  memcpy(&h, buf, sizeof h);
  if (h.magic != kSnapMagic || h.abi != LBFT_ABI_VERSION) return set_error(LBFT_ERR_INVALID, "not a snapshot of this library version");
  if (bytes != need || h.num_instances != s->I || h.num_nodes != s->N || h.total_words != s->P.L.total_words ||
      h.max_clock != s->P.max_clock || h.config_digest != config_digest(s))
    return set_error(LBFT_ERR_INVALID, "the snapshot was taken from a differently configured simulator");
  if (int r = need_idle(s)) return r;
  CUDA_TRY(cudaSetDevice(s->device));
  CUDA_TRY(cudaMemcpy(s->d_state, static_cast<const char*>(buf) + sizeof h, state_bytes(s), cudaMemcpyHostToDevice));
  s->started = true;   // the next lbft_run_until restores the instances from their save areas
  s->uploaded = true;  // the seeds are not needed any more
  s->ran = false;
  s->downloaded = false;
  s->last_stop = h.last_stop;
  return LBFT_OK;
}

static int need_results(lbft_sim* s, const void* out) {
  if (!s || !out) return set_error(LBFT_ERR_INVALID, "NULL argument");
  // (while an lbft_run_async is in flight the getters keep serving the previous run's results: they live in the
  // other set of host mirrors)
  if (!s->downloaded) return set_error(LBFT_ERR_STATE, "results are not available: call lbft_run (or lbft_download) first");
  return LBFT_OK;
}
int lbft_commit_counts(lbft_sim* s, uint32_t* out) {
  if (int r = need_results(s, out)) return r;
  memcpy(out, s->res[s->done].commit_counts, (size_t)s->I * s->N * sizeof(uint32_t));
  return LBFT_OK;
}
int lbft_last_states(lbft_sim* s, uint64_t* out) {
  if (int r = need_results(s, out)) return r;
  memcpy(out, s->res[s->done].last_state, (size_t)s->I * s->N * sizeof(uint64_t));
  return LBFT_OK;
}
int lbft_counters(lbft_sim* s, lbft_instance_counters* out) {
  if (int r = need_results(s, out)) return r;
  memcpy(out, s->res[s->done].counters, (size_t)s->I * 12 * sizeof(uint32_t));
  return LBFT_OK;
}
int lbft_active_rounds(lbft_sim* s, uint32_t* out) {
  if (int r = need_results(s, out)) return r;
  memcpy(out, s->res[s->done].rounds, (size_t)s->I * sizeof(uint32_t));  // == lbft_instance_counters.max_active_round
  return LBFT_OK;
}
int lbft_status(lbft_sim* s, uint32_t* out) {
  if (int r = need_results(s, out)) return r;
  memcpy(out, s->res[s->done].status, (size_t)s->I * sizeof(uint32_t));
  return LBFT_OK;
}
int lbft_timing_info(lbft_sim* s, lbft_timing* out) {
  if (!s || !out) return set_error(LBFT_ERR_INVALID, "NULL argument");
  *out = s->timing;
  return LBFT_OK;
}
int lbft_kernel_info(lbft_sim* s, char* buf, size_t cap) {
  if (!s || !buf || cap == 0) return set_error(LBFT_ERR_INVALID, "NULL argument");
  snprintf(buf, cap, "%s", kernel_name(s).c_str());
  return LBFT_OK;
}
int lbft_memory_info(lbft_sim* s, uint64_t* device_bytes, uint32_t* words_per_instance) {
  if (!s) return set_error(LBFT_ERR_INVALID, "NULL argument");
  if (device_bytes) *device_bytes = s->device_bytes;
  if (words_per_instance) *words_per_instance = s->P.L.total_words;
  return LBFT_OK;
}

// committed_history() of one node: walk the instance's chain table backwards from the node's last
// committed round (every commit extends the previous one by exactly one block,
// simulated_context.rs:172-174, so the log is the ancestor chain of the last committed block).
int lbft_commit_log(lbft_sim* s, uint32_t instance, uint32_t node, lbft_commit* out, size_t cap, size_t* n) {
  if (!s || !n) return set_error(LBFT_ERR_INVALID, "NULL argument");
  if (!s->downloaded) return set_error(LBFT_ERR_STATE, "results are not available: call lbft_run first");
  if (instance >= s->I || node >= s->N) return set_error(LBFT_ERR_INVALID, "instance/node out of range");
  if (cap && !out) return set_error(LBFT_ERR_INVALID, "out must not be NULL when cap > 0");
  if (int r = need_idle(s)) return r;
  CUDA_TRY(cudaSetDevice(s->device));
  const Layout& L = s->P.L;
  std::vector<uint32_t> chain(2 * (size_t)L.round_cap);
  const uint32_t S = s->stride, tile = instance / S, lane = instance % S;
  const uint32_t* src = s->d_state + ((size_t)tile * L.total_words + L.chain_base) * S + lane;
  CUDA_TRY(cudaMemcpy2D(chain.data(), sizeof(uint32_t), src, S * sizeof(uint32_t), sizeof(uint32_t), chain.size(), cudaMemcpyDeviceToHost));
  uint32_t lc = s->res[s->done].lc_round[(size_t)instance * s->N + node];
  uint32_t count = s->res[s->done].commit_counts[(size_t)instance * s->N + node];
  // epochs > 1: the parent of an epoch's first block is the block whose state is the epoch's initial state
  std::vector<uint32_t> einit(L.epochs, 0);
  if (L.epochs > 1)
    CUDA_TRY(cudaMemcpy2D(einit.data(), sizeof(uint32_t), s->d_state + ((size_t)tile * L.total_words + L.einit_base) * S + lane,
                          S * sizeof(uint32_t), sizeof(uint32_t), L.epochs, cudaMemcpyDeviceToHost));
  std::vector<lbft_commit> log(count);
  uint32_t i = count;
  for (uint32_t r = lc; r != 0 && i > 0;) {
    if (r >= L.round_cap) return set_error(LBFT_ERR_STATE, "corrupt chain table");
    --i;
    log[i].proposer = s->hs.leader[r % L.rspan];
    log[i].index = chain[2 * r] >> 16;
    log[i].time = (int64_t)(int32_t)chain[2 * r + 1];
    const uint32_t p = chain[2 * r] & 0xffffu, e = r / L.rspan;
    r = p ? e * L.rspan + p : einit[e];
  }
  if (i != 0) return set_error(LBFT_ERR_STATE, "chain shorter than the commit count");
  *n = count;
  for (size_t k = 0; k < count && k < cap; k++) out[k] = log[k];
  return LBFT_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Bulk read-out of the commit logs: one device pass + one device->host copy for the whole batch
// (committed_history() of every context, simulated_context.rs:98-100; lbft_commit_log does one strided copy per
// (instance, node) and is meant for spot checks).
// Every commit extends the previous one by exactly one block (simulated_context.rs:172-174), so a node's log is the
// ancestor chain of its last committed block; the kernel lays out the LONGEST log of each instance in commit order
// and verifies that every other node's last committed block lies on it at depth == its commit count (SURVEY App.
// C.3).  Instances where that does not hold are counted in *bad.
// ---------------------------------------------------------------------------------------------
__global__ void lbft_commit_logs_kernel(const __grid_constant__ Params P, uint32_t stride, lbft_commit* out, uint32_t cap, uint32_t* bad) {
  const uint32_t inst = blockIdx.x * blockDim.x + threadIdx.x;
  if (inst >= P.num_instances) return;
  const Layout& L = P.L;
  const uint32_t N = L.num_nodes, tile = inst / stride, lane = inst % stride;
  const uint32_t* tb = P.state + (size_t)tile * L.total_words * stride + lane;
  const uint32_t* cc = P.out_commit_counts + (size_t)inst * N;
  const uint32_t* lc = P.out_lc_round + (size_t)inst * N;
  uint32_t best = 0;
  for (uint32_t n = 1; n < N; n++)
    if (cc[n] > cc[best]) best = n;
  uint32_t k = cc[best], r = lc[best], matched = 0;
  lbft_commit* row = out + (size_t)inst * cap;
  while (r != 0 && k > 0) {
    for (uint32_t n = 0; n < N; n++)
      if (cc[n] == k) matched += lc[n] == r ? 1u : 0x10000u;
    --k;
    const uint32_t c0 = tb[(size_t)(L.chain_base + 2 * r) * stride];
    if (k < cap) {
      lbft_commit e;
      e.proposer = P.leader[r % L.rspan];
      e.index = c0 >> 16;
      e.time = (int64_t)(int32_t)tb[(size_t)(L.chain_base + 2 * r + 1) * stride];
      row[k] = e;
    }
    const uint32_t p = c0 & 0xffffu, ep = r / L.rspan;
    r = p ? ep * L.rspan + p : (L.epochs > 1 ? tb[(size_t)(L.einit_base + ep) * stride] : 0u);
  }
  uint32_t empty = 0;
  for (uint32_t n = 0; n < N; n++) empty += cc[n] == 0 ? (lc[n] == 0 ? 1u : 0x10000u) : 0u;
  if (r != 0 || k != 0 || matched + empty != N) atomicAdd(bad, 1u);
}

int lbft_commit_logs(lbft_sim* s, lbft_commit* out, size_t cap, uint32_t* lens) {
  if (!s || !out || cap == 0) return set_error(LBFT_ERR_INVALID, "out must not be NULL and cap must be > 0");
  if (!s->downloaded) return set_error(LBFT_ERR_STATE, "results are not available: call lbft_run first");
  if (cap > 0xffffu) return set_error(LBFT_ERR_INVALID, "cap must be <= 65535 rows per instance");
  if (int r = need_idle(s)) return r;
  CUDA_TRY(cudaSetDevice(s->device));
  if (cap > s->logs_cap) {
    cudaFree(s->d_logs);
    s->d_logs = nullptr;
    s->logs_cap = 0;
    cudaError_t e = cudaMalloc((void**)&s->d_logs, (size_t)s->I * cap * sizeof(lbft_commit));
    if (e != cudaSuccess) return set_error(LBFT_ERR_NOMEM, std::string("commit-log buffer: ") + cudaGetErrorString(e));
    s->logs_cap = cap;
  }
  // rows beyond a log's length are zero
  CUDA_TRY(cudaMemsetAsync(s->d_logs, 0, (size_t)s->I * cap * sizeof(lbft_commit), s->stream));
  CUDA_TRY(cudaMemsetAsync(s->d_error, 0, sizeof(uint32_t), s->stream));
  lbft_commit_logs_kernel<<<(s->I + 127) / 128, 128, 0, s->stream>>>(s->P, s->stride, s->d_logs, (uint32_t)cap, s->d_error);
  CUDA_TRY(cudaGetLastError());
  uint32_t bad = 0;
  CUDA_TRY(cudaMemcpyAsync(out, s->d_logs, (size_t)s->I * cap * sizeof(lbft_commit), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(&bad, s->d_error, sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (lens) memcpy(lens, s->res[s->done].commit_counts, (size_t)s->I * s->N * sizeof(uint32_t));
  if (bad) {
    char buf[160];
    snprintf(buf, sizeof buf, "%u instance(s) have node logs that are not prefixes of one chain: read them with lbft_commit_log", bad);
    return set_error(LBFT_ERR_STATE, buf);
  }
  return LBFT_OK;
}

extern "C" {

int lbft_round_switches(lbft_sim* s, uint32_t instance, lbft_round_switch* out, size_t cap, size_t* n) {
  if (!s || !n) return set_error(LBFT_ERR_INVALID, "NULL argument");
  if (!s->P.record_rs) return set_error(LBFT_ERR_STATE, "round switches were not recorded: set LBFT_FLAG_ROUND_SWITCHES in lbft_config.flags");
  if (!s->downloaded) return set_error(LBFT_ERR_STATE, "results are not available: call lbft_run first");
  if (instance >= s->I) return set_error(LBFT_ERR_INVALID, "instance out of range");
  if (cap && !out) return set_error(LBFT_ERR_INVALID, "out must not be NULL when cap > 0");
  CUDA_TRY(cudaSetDevice(s->device));
  const Layout& L = s->P.L;
  const uint32_t row = L.round_cap + 1;
  std::vector<uint32_t> table((size_t)s->N * row);
  const uint32_t S = s->stride, tile = instance / S, lane = instance % S;
  const uint32_t* src = s->d_state + ((size_t)tile * L.total_words + rs_table_base(L)) * S + lane;
  CUDA_TRY(cudaMemcpy2D(table.data(), sizeof(uint32_t), src, S * sizeof(uint32_t), sizeof(uint32_t), table.size(), cudaMemcpyDeviceToHost));
  size_t k = 0;
  for (uint32_t node = 0; node < s->N; node++)
    for (uint32_t r = 1; r < row; r++) {  // slot 0 is the per-node maximum, not a switch
      const uint32_t w = table[(size_t)node * row + r];
      if (!w) continue;
      if (k < cap) out[k] = lbft_round_switch{node, r, (int64_t)(w - 1u)};
      k++;
    }
  *n = k;
  return LBFT_OK;
}

void lbft_destroy(lbft_sim* s) { free_all(s); }

}  // extern "C"
