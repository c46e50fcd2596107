#!/usr/bin/env python
"""bench.py — simulated consensus rounds/sec of the batched LibraBFTv2 event loop (BASELINE.json metric).

A "step" is one pass of the hot path over one batch: `Simulator::new` + `loop_until(max_clock)` for every
instance of the batch.  The default workload is BASELINE.json configs[2] (SURVEY §8d.3): 65 536 instances x 4
authors per GPU, LogNormal(10, 4) delays, max_clock = 1000; `--config K` (K = 1..5, SURVEY §8d inputs 1-5) selects
another BASELINE configuration as the bench line.  Each step uses fresh seeds.

  value     rounds/s with the seeds already resident in HBM (kernel only, CUDA events, max over ranks)
  e2e       rounds/s through the public API with HOST buffers: seeds host->device, kernel, summaries device->host
            (commit counts, state keys, rounds, status land in caller-owned arrays), every step
  roofline  algorithmic bytes (SURVEY §8d formula over the run's own event counters) / kernel time vs the measured
            HBM copy peak; the measured DRAM traffic (ncu) and its own rate are reported next to it
  parity    EVERY instance of the last timed batch is compared with the CPU oracle (commit counts, state keys,
            event/RNG counters) outside the timed region ("checked N of N"; a bounded sample only where the oracle
            would need more than a minute, and then it says so)
  cpu_baseline  the CPU oracle (oracle/, a C++ restatement pinned by the reference goldens — no Rust toolchain
            exists here; -O3 -march=native build made on this machine) timed on the host cores on a bounded sample
  configs   (default run, 1 GPU) the other four BASELINE configurations, each measured and parity-checked the same way

`--impl reference` times that CPU implementation alone (all host threads) on the same metric/config.
`--dump-outputs DIR` writes the results of the last timed step as .npy files (see dump_outputs), so that two builds run
with the same arguments, hence on the same seeds, can be compared output for output.
Multi-GPU: one process per GPU under torchrun through `ShardedBatchSimulator`: instances sharded with no data-path
collective; one NCCL all-gather of the per-instance summaries at the end of every step.  "scaling": "weak" (the
configuration's batch per GPU) unless `--scaling strong` (the configuration's batch split over the GPUs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "simulated consensus rounds/sec (whole box)"
UNIT = "rounds/s"
W64 = [1 + (i % 3) for i in range(64)]
SILENT64 = [1 if i % 3 == 0 and i <= 60 else 0 for i in range(64)]

# BASELINE.json configs[0..4] as SURVEY §8(d) fixes their inputs.  `kw` are lbft_config fields in the keyword form
# shared by the product mirror (make_sim below) and the oracle wrapper (tests.support.make_config).
CONFIGS = {
    1: dict(instances=1, nodes=3, max_clock=3000, base_seed=52, kw=dict(delay_variance=0.0),
            text="1 instance x 3 authors, fixed 10 ms delay (LogNormal(10, 0)), max_clock=3000 (>100 rounds) (BASELINE configs[0], SURVEY 8d.1)"),
    2: dict(instances=1024, nodes=4, max_clock=1000, base_seed=52, kw=dict(delay_kind=1, delay_lo=5, delay_hi=15),
            text="1 024 instances x 4 authors, uniform[5,15] ms delay, max_clock=1000 (BASELINE configs[1], SURVEY 8d.2)"),
    3: dict(instances=65536, nodes=4, max_clock=1000, base_seed=52, kw={},
            text="65 536 instances x 4 authors per GPU, LogNormal(10,4) delay, max_clock=1000, delta=20 gamma=2 lambda=0.5 "
                 "(BASELINE configs[2], SURVEY 8d.3)"),
    4: dict(instances=8192, nodes=64, max_clock=1000, base_seed=52, kw=dict(voting_rights=W64, silent=SILENT64),
            text="8 192 instances x 64 authors, voting rights 1+(i mod 3), 21 silent nodes, LogNormal(10,4), max_clock=1000 "
                 "(BASELINE configs[3], SURVEY 8d.4)"),
    5: dict(instances=16384, nodes=7, max_clock=1000, base_seed=1, kw=dict(partition_windows=4, partition_max_len=150),
            text="16 384 instances x 7 authors, 4 random partition windows (<=150 ms) per instance, LogNormal(10,4), max_clock=1000, "
                 "base seeds swept per step (BASELINE configs[4], SURVEY 8d.5)"),
}
ORACLE_PARITY_BUDGET_S = 45.0   # full-batch compare whenever the oracle needs less than this; else a strided sample


def make_sim(seeds, nodes, device=0, **kw):
    """A BatchSimulator from the keyword form of an lbft_config."""
    from librabft_simulator_b200 import BatchSimulator, NodeConfig, RandomDelay
    kw = dict(kw)
    delay = RandomDelay.new(kw.pop("delay_mean", 10.0), kw.pop("delay_variance", 4.0))
    if "delay_lo" in kw:
        delay = RandomDelay.uniform(kw.pop("delay_lo"), kw.pop("delay_hi"))
        kw.pop("delay_kind", None)
    return BatchSimulator(seeds, nodes, delay, NodeConfig(), 30000, device=device, **kw)


def algorithmic_bytes(counters, n_nodes):
    """SURVEY.md §8(d): Bytes = P*(2*S_node + S_hdr) + P_notify*S_notif + Q*S_hdr + Q_notify*S_notif."""
    s_hdr, s_node, s_notif = 16, 208 + 12 * n_nodes, 40 + 10 * n_nodes
    c = counters.astype(np.float64)
    p = c[:, 0:4].sum()
    p_notify = c[:, 0].sum()
    q = c[:, 5].sum()
    q_notify = c[:, 9].sum()
    return p * (2 * s_node + s_hdr) + p_notify * s_notif + q * s_hdr + q_notify * s_notif


def effective_cores():
    """Host threads we can actually use: CPU affinity capped by the cgroup CPU quota (the GPU boxes expose 128
    logical CPUs but grant 16 CPUs of quota; oversubscribing only adds throttling)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def ncu_traffic_bytes(config_id, per_gpu, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the event-loop kernel, from the committed ncu
    --set full capture (profiles/traffic.json: one entry per (config, kernel)); None if there is no matching capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        for e in t.get("captures", []):
            if e.get("config") == config_id and e.get("instances") == per_gpu and e.get("kernel") == kernel:
                return e["dram_bytes_per_launch"], e.get("source")
    except Exception:
        pass
    return None, None


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smmax, reasons = [], [], set()
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smmax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smmax) if smmax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def step_seeds(cfg, step, first_instance, count):
    """Instance i of the whole job uses seed base_seed + i; every step moves on to a fresh block of seeds (for config 5
    that is the base-seed sweep of SURVEY 8d.5)."""
    first = cfg["base_seed"] + step * (1 << 24) + first_instance
    return np.arange(first, first + count, dtype=np.uint64)


# ------------------------------------------------------------------------------------------------------------
# CPU side: oracle timing (cpu_baseline, --impl reference) and the parity check
# ------------------------------------------------------------------------------------------------------------
_ORACLE = {}


def get_oracle():
    """The -O3 -march=native build of the oracle, compiled on this machine (BASELINE.md §2); test infrastructure, used
    here only as the timed CPU baseline and as the checker."""
    if "o" not in _ORACLE:
        from tests.support import Oracle
        _ORACLE["o"] = Oracle(native=True)
    return _ORACLE["o"]


def run_cpu_sample(cfg, seeds, threads):
    oracle = get_oracle()   # (built on first use: outside the timed region)
    t0 = time.perf_counter()
    res = oracle.run(seeds, cfg["nodes"], cfg["max_clock"], threads=threads, **cfg["kw"])
    dt = time.perf_counter() - t0
    return float(res.counters[:, 6].sum()), dt, res


def oracle_seconds_per_instance(cfg, threads):
    """Probe: wall seconds per instance with `threads` threads busy (one instance per task)."""
    n = min(cfg["instances"], 2 * threads)
    _, dt, _ = run_cpu_sample(cfg, step_seeds(cfg, 4000, 0, n), threads)   # also warms the thread pool / page cache
    for _ in range(2):  # too short to extrapolate from (start-up costs, scheduler noise): grow the sample to about a second
        if dt >= 0.5 or n >= cfg["instances"]:
            break
        n = min(cfg["instances"], max(2 * n, int(n * 1.0 / max(dt, 1e-4))))
        _, dt, _ = run_cpu_sample(cfg, step_seeds(cfg, 4100, 0, n), threads)
    return dt / n


def parity_and_cpu_baseline(cfg, seeds, gpu, budget_s=ORACLE_PARITY_BUDGET_S):
    """Compare the GPU batch `gpu` (arrays for `seeds`) with the oracle — every instance when the oracle finishes within
    `budget_s`, else a strided sample of the size that does — and report the oracle's own speed on that run as the CPU
    baseline of the configuration.  Outside every timed region."""
    threads = effective_cores()
    per_inst = oracle_seconds_per_instance(cfg, threads)
    total = len(seeds)
    n = total if per_inst * total <= budget_s else int(max(threads, min(total, budget_s / per_inst)))
    idx = np.arange(total) if n == total else np.unique(np.linspace(0, total - 1, n).astype(np.int64))
    rounds, dt, ref = run_cpu_sample(cfg, seeds[idx], threads)
    bad = np.zeros(len(idx), dtype=bool)
    bad |= (ref.commit_counts != gpu["commit_counts"][idx]).any(axis=1)
    bad |= (ref.last_states != gpu["last_states"][idx]).any(axis=1)
    bad |= (ref.counters[:, :8] != gpu["counters"][idx, :8]).any(axis=1)
    bad |= ref.counters[:, 9] != gpu["counters"][idx, 9]
    parity = {"checked": int(len(idx)), "of": int(total), "mismatches": int(bad.sum()), "ok": bool(not bad.any()),
              "compared": "commit counts, state keys (SipHash of the commit log), counters[0:8] + scheduled notifications, per instance",
              "oracle_seconds": dt}
    if bad.any():
        parity["first_mismatch_seed"] = int(seeds[idx][np.argmax(bad)])
    base = {"value": rounds / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d of %d instances x %d authors, max_clock=%d, %.1f s wall, %d threads; C++ oracle restating the Rust "
                      "reference (no Rust toolchain), %s build, pinned by the reference goldens"
                      % (len(idx), total, cfg["nodes"], cfg["max_clock"], dt, threads, get_oracle().build_flags)}
    return parity, base


def run_reference_arm(args, cfg, rank):
    """`--impl reference`: the reference's CPU implementation of the path (here: the C++ oracle port, because the
    Rust reference cannot be built in this image) on all host threads; rank 0 only."""
    if rank != 0:
        return
    threads = effective_cores()
    per_gpu = cfg["instances"]
    per_inst = oracle_seconds_per_instance(cfg, threads)
    budget = min(120.0 / max(1, args.steps + args.warmup), 20.0)  # bounded sample per step: the whole run ends within minutes
    count = int(max(min(per_gpu, threads), min(per_gpu, budget / max(per_inst, 1e-9))))
    for w in range(args.warmup):
        run_cpu_sample(cfg, step_seeds(cfg, 1000 + w, 0, count), threads)
    rounds_total, t_total = 0.0, 0.0
    for s in range(args.steps):
        r, dt, _ = run_cpu_sample(cfg, step_seeds(cfg, s, 0, count), threads)
        rounds_total += r
        t_total += dt
    value = rounds_total / t_total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": cfg["text"] + "; reference arm steps over a bounded sample of %d instances" % count,
                   "seeds": "base_seed %d + instance" % cfg["base_seed"]},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d instances per step, %d threads; C++ oracle port of the Rust reference (reference not "
                                   "buildable here: no cargo/rustc), %s build" % (count, threads, get_oracle().build_flags)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------
def gpu_arrays(res):
    return {"commit_counts": res.commit_counts, "last_states": res.last_committed_states, "counters": res.counters}


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(res, out_dir, limit_bytes=DUMP_LIMIT_BYTES):
    """Write what a caller of the timed path receives for one batch (a BatchResult) to out_dir/<name>.npy, all float64:
    commit_counts [I][N]; last_committed_states_hi and _lo [I][N], the upper and lower 32 bits of the 64-bit state keys (each
    exact in float64); active_rounds [I]; status [I]; counters [I][12]; and instance [I], the batch index of each row.  When
    all of it would exceed limit_bytes, the rows are a fixed, seeded sample of the instances, the same one on every run."""
    states = np.asarray(res.last_committed_states, dtype=np.uint64)
    arrays = {"commit_counts": res.commit_counts, "last_committed_states_hi": states >> np.uint64(32),
              "last_committed_states_lo": states & np.uint64(0xFFFFFFFF), "active_rounds": res.active_rounds,
              "status": res.status, "counters": res.counters}
    total = len(states)
    row_bytes = 8 * (1 + sum(int(np.prod(np.shape(a)[1:])) for a in arrays.values()))
    rows = np.arange(total)
    if total * row_bytes > limit_bytes:
        keep = (limit_bytes - 4096) // row_bytes   # 4 KB of headroom for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(total, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "instance.npy"), rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a)[rows].astype(np.float64))


def roofline_block(cfg_id, cfg, per_gpu, counters, kernel_ms, kernel_name):
    peak, peak_src = measured_peak_gbs()
    bytes_launch = algorithmic_bytes(counters, cfg["nodes"])
    achieved = bytes_launch / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic_bytes(cfg_id, per_gpu, kernel_name)
    block = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
             "traffic_source": traffic_src, "peak_source": peak_src, "kernel": kernel_name, "kernel_ms": kernel_ms,
             "algorithmic_bytes_per_launch": bytes_launch,
             "events_per_s": float(counters[:, 0:4].sum()) / (kernel_ms * 1e-3),
             "note": "achieved/frac are the ALGORITHMIC (layout-independent) bytes of SURVEY 8d over the kernel time; the kernel is "
                     "issue/latency-bound, its real DRAM traffic is `traffic` (ncu) = dram_achieved GB/s"}
    if traffic:
        block["dram_achieved"] = traffic / (kernel_ms * 1e-3) / 1e9
        block["dram_frac"] = block["dram_achieved"] / peak
    return block


def measure_side_config(cfg_id, device, steps, warmup):
    """One of the non-headline BASELINE configurations on one GPU: kernel time (CUDA events, seeds resident), e2e time
    (host buffers), full parity and the CPU baseline.  Used for the `configs` block of the default line."""
    import torch
    cfg = CONFIGS[cfg_id]
    I = cfg["instances"]
    sim = make_sim(step_seeds(cfg, 0, 0, I), cfg["nodes"], device=device, **cfg["kw"])
    sim.create(cfg["max_clock"])
    for w in range(warmup):
        sim.set_seeds(step_seeds(cfg, 10000 + w, 0, I))
        sim.run(strict=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_rounds = 0.0
    for r in sim.run_stream((step_seeds(cfg, s, 0, I) for s in range(steps)), strict=False):
        e2e_rounds += float(r.active_rounds.sum())
    e2e_s = time.perf_counter() - t0
    kms, rounds, res, seeds = [], 0.0, None, None
    for s in range(steps):
        seeds = step_seeds(cfg, 100 + s, 0, I)
        sim.set_seeds(seeds)
        sim.upload()
        sim.run_device()
        kms.append(float(sim.timing.sim_ms))
        res = sim.download(strict=False)
        rounds += float(res.active_rounds.sum())
    k_ms = float(np.mean(kms))
    kernel = sim.kernel_info()
    parity, base = parity_and_cpu_baseline(cfg, seeds, gpu_arrays(res))
    out = {"workload": cfg["text"], "kernel": kernel, "kernel_ms": k_ms, "value": rounds / (sum(kms) * 1e-3), "unit": UNIT,
           "e2e": e2e_rounds / e2e_s, "steps": steps, "warmup": warmup,
           "events_per_s": float(res.counters[:, 0:4].sum()) / (k_ms * 1e-3),
           "roofline": roofline_block(cfg_id, cfg, I, res.counters, k_ms, kernel),
           "flagged_instances": int(((res.status & 0x9E) != 0).sum()),
           "parity": parity, "cpu_baseline": base, "e2e_over_cpu": (e2e_rounds / e2e_s) / base["value"]}
    sim.close()
    return out


_REAL_STDOUT = None


def quiet_stdout():
    """Route everything libraries print on stdout (e.g. the NCCL version banner) to stderr, so that the ONE JSON line
    the driver parses is the only thing on stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from, which may be read-only
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS), help="BASELINE.json configs[K-1] (default 3 = the metric's)")
    ap.add_argument("--instances", type=int, default=0, help="override the instances per GPU of the configuration")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the configuration's batch per GPU; strong: the configuration's batch split over the GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle (no parity check, no cpu_baseline)")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config block of the default line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step (rank 0's shard) to "
                                                          "DIR/<name>.npy as float64, at most 64 MB (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU path; the reference arm times a machine-dependent sample")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = dict(CONFIGS[args.config])
    if args.instances:
        cfg["instances"] = args.instances
        cfg["text"] += " [instances per GPU overridden: %d]" % args.instances
    if args.impl == "reference":
        run_reference_arm(args, cfg, rank)
        return

    import torch
    import torch.distributed as dist
    from librabft_simulator_b200 import ShardedBatchSimulator

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    nodes, max_clock = cfg["nodes"], cfg["max_clock"]
    total = cfg["instances"] * world if args.scaling == "weak" else cfg["instances"] // world * world
    per_gpu = total // world

    def job_seeds(step):
        return step_seeds(cfg, step, 0, total)

    def make_local(shard):
        return make_sim(shard, nodes, device=local_rank, **cfg["kw"])

    sharded = ShardedBatchSimulator(job_seeds(0), nodes, rank=rank, world=world, dist=dist if distributed else None,
                                    device=local_rank, make_local=make_local)
    sharded.create(max_clock)
    sim = sharded.local
    dev_bytes, words_per_inst = sim.memory_info()
    kernel = sim.kernel_info()

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    # nvidia-smi needs a moment before its first sample: start it ahead of the warm-up (also load) so that the short timed
    # region is covered
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---------------- warm-up (both legs) ----------------
    for w in range(args.warmup):
        sharded.set_seeds(job_seeds(10000 + w))
        sharded.run(strict=False)
    barrier()

    # ---------------- e2e leg: host buffers in, host results out, every step ----------------
    e2e_rounds = 0.0
    barrier()
    t0 = time.perf_counter()
    # One run is always in flight (ShardedBatchSimulator.run_stream = lbft_run_async / lbft_wait): every step copies its seeds
    # host->device from the pinned staging buffer and its summaries device->host into caller-owned arrays, and is
    # all-gathered; the staging of step k + 1 and the host-side copies of step k overlap a kernel.
    for res in sharded.run_stream((job_seeds(s) for s in range(args.steps)), strict=False):
        e2e_rounds += float(res.local.active_rounds.sum())
    barrier()
    e2e_seconds = time.perf_counter() - t0
    h2d_bytes, d2h_bytes = int(sim.timing.h2d_bytes), int(sim.timing.d2h_bytes)

    # ---------------- value leg: inputs resident in HBM, device-timed kernel ----------------
    kernel_ms, rounds_dev, last, last_seeds, flagged = [], 0.0, None, None, 0
    barrier()
    for s in range(args.steps):
        last_seeds = job_seeds(100 + s)[sharded.lo:sharded.hi]
        sim.set_seeds(last_seeds)
        sim.upload()                                      # outside the timed region
        sim.run_device()                                  # CUDA events on the launching stream around the kernel
        kernel_ms.append(float(sim.timing.sim_ms))
        last = sim.download(strict=False)
        sharded.gather(last)
        rounds_dev += float(last.active_rounds.sum())
        flagged += int(((last.status & 0x9E) != 0).sum())  # any LBFT_ST_ERROR_MASK bit (capacity / invariant / epoch)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(last, args.dump_outputs)

    dev_seconds = sum(kernel_ms) / 1e3
    stats = torch.tensor([dev_seconds, e2e_seconds], dtype=torch.float64, device="cuda")
    sums = torch.tensor([rounds_dev, e2e_rounds], dtype=torch.float64, device="cuda")
    if distributed:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)     # max over ranks
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)      # whole-job totals
    dev_seconds, e2e_seconds = stats.tolist()
    rounds_dev, e2e_rounds = sums.tolist()

    if rank == 0:
        value = rounds_dev / dev_seconds
        k_ms = float(np.mean(kernel_ms))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dev_seconds / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": {"workload": cfg["text"], "baseline_config": args.config,
                       "seeds": "base_seed %d + instance, fresh block per step" % cfg["base_seed"],
                       "instances_total": total, "instances_per_gpu": per_gpu,
                       "l2": "state working set %.0f MB per GPU (126 MB L2); every step re-initialises it" % (dev_bytes / 1e6),
                       "parallelism": "instances sharded over %d GPU(s) (ShardedBatchSimulator); one NCCL all-gather of {commit counts, "
                                      "state keys, rounds} per step" % world},
            "e2e": {"value": e2e_rounds / e2e_seconds, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": 1e3 * e2e_seconds / args.steps,
                    "returns": "commit counts [I][N], state keys [I][N], rounds [I], status [I] in caller-owned host arrays",
                    "pipeline": "run_stream: one run in flight per GPU (lbft_run_async / lbft_wait, double-buffered pinned staging)"},
            "gpu_launches": args.steps * 2,
            "roofline": roofline_block(args.config, cfg, per_gpu, last.counters, k_ms, kernel),
            "clocks": clocks,
            "state_bytes_per_instance": words_per_inst * 4,
            "flagged_instances": flagged,  # instances (rank 0, value leg) that hit a capacity/invariant flag: expected 0
        }
        if not args.no_cpu_baseline:
            # parity of the LAST TIMED batch (rank 0's shard), every instance, against the oracle; its speed = cpu_baseline
            parity, base = parity_and_cpu_baseline(cfg, last_seeds, gpu_arrays(last))
            line["parity"] = parity
            line["cpu_baseline"] = base
            if world == 1 and args.config == 3 and not args.no_configs and not args.instances:
                sim.close()
                side = {}
                for k in (1, 2, 4, 5):
                    side[str(k)] = measure_side_config(k, local_rank, args.steps, args.warmup)
                me = {"workload": cfg["text"], "kernel": kernel, "kernel_ms": k_ms, "value": value, "unit": UNIT,
                      "e2e": line["e2e"]["value"], "events_per_s": line["roofline"]["events_per_s"], "roofline": line["roofline"],
                      "flagged_instances": flagged, "parity": parity, "cpu_baseline": base,
                      "e2e_over_cpu": line["e2e"]["value"] / base["value"]}
                side["3"] = me
                line["configs"] = {k: side[k] for k in sorted(side)}
        emit(line)
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
