#!/usr/bin/env python
"""One sweep handle against the same parameter sets run as one plain handle each (one B200, one process).

  (a) 64 sets x 1 024 seeds, 4 authors, max_clock 1000: one lbft_create_sweep handle vs 64 lbft_create handles of 1 024
      instances run one after another;
  (b) the same at 7 authors, 16 sets x 1 024 seeds;
  (c) the plain 65 536 x 4 handle of bench.py's default line, as the reference point.

Kernel time is lbft_timing_info's CUDA-event sim_ms (summed over the plain handles); wall time is the host clock around
lbft_run calls that end in a stream synchronise (summed likewise; handle creation excluded).  Every shape is run once as a
warm-up, then --reps times; the medians are reported.  Every timed sweep is checked for parity, instance by instance,
against the outputs of the plain handles (commit counts, state keys, counters, status, active rounds).  The card's name
and power limit are read in the same process.  Usage: python tools/measure_sweep.py [--reps 5] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from librabft_simulator_b200 import BatchSimulator, NodeConfig, ParamSet, RandomDelay  # noqa: E402


def grid(n, num_nodes):
    """Delay mean x variance x delta x gamma x lambda, a few uniform-delay sets and a few with one silent node."""
    out = []
    for k in range(n):
        d = RandomDelay.new(6.0 + 2.0 * (k % 8), [0.0, 1.0, 4.0, 9.0][(k // 8) % 4])
        if k % 13 == 5:
            d = RandomDelay.uniform(3 + k % 4, 12 + k % 7)
        nc = NodeConfig(100000, [15, 20, 30, 40][k % 4], [1.5, 2.0][(k // 2) % 2], [0.5, 1.0][(k // 16) % 2])
        silent = [0] * (num_nodes - 1) + [1] if k % 11 == 3 else None
        out.append(ParamSet(d, nc, silent))
    return out


def outputs(res):
    c = res.counters
    return [res.commit_counts, res.last_committed_states, c[:, :8], c[:, 9], res.status, res.active_rounds]


def timed(sim, reps):
    kern, wall, res = [], [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        res = sim.run()
        wall.append((time.perf_counter() - t0) * 1e3)
        kern.append(sim.timing.sim_ms)
    return kern, wall, res


def compare(num_nodes, num_sets, per_set, reps, max_clock=1000):
    sets = grid(num_sets, num_nodes)
    I = num_sets * per_set
    set_of = np.random.default_rng(num_nodes).permutation(np.arange(I) % num_sets).astype(np.uint32)
    seeds = np.arange(1, I + 1, dtype=np.uint64)
    sweep = BatchSimulator(seeds, num_nodes, param_sets=sets, set_index=set_of).create(max_clock)
    sweep.run()  # warm-up
    s_kern, s_wall, s_res = timed(sweep, reps)
    plain = []
    for k, p in enumerate(sets):
        sim = BatchSimulator(seeds[set_of == k], num_nodes, p.network_delay, p.node_config, silent=p.silent).create(max_clock)
        sim.run()  # warm-up
        plain.append(sim)
    p_kern, p_wall = np.zeros(reps), np.zeros(reps)
    p_res = []
    for sim in plain:
        k, w, r = timed(sim, reps)
        p_kern += k
        p_wall += w
        p_res.append(r)
    checked = 0
    for k, r in enumerate(p_res):
        sel = set_of == k
        for a, b in zip(outputs(s_res), outputs(r)):
            if not np.array_equal(a[sel], b):
                raise SystemExit("parity failure: set %d of the %d-author sweep differs from its plain handle" % (k, num_nodes))
        checked += int(sel.sum())
    kernel_name = sweep.kernel_info()
    plain_kernel = plain[0].kernel_info()
    rounds = int(s_res.active_rounds.astype(np.int64).sum())
    for sim in plain + [sweep]:
        sim.close()
    sk, sw, pk, pw = float(np.median(s_kern)), float(np.median(s_wall)), float(np.median(p_kern)), float(np.median(p_wall))
    return {"num_nodes": num_nodes, "sets": num_sets, "seeds_per_set": per_set, "instances": I, "max_clock": max_clock,
            "sweep_kernel": kernel_name, "plain_kernel": plain_kernel,
            "sweep_kernel_ms": sk, "sweep_wall_ms": sw, "plain_handles_kernel_ms_sum": pk, "plain_handles_wall_ms_sum": pw,
            "kernel_speedup": pk / sk, "wall_speedup": pw / sw, "sweep_rounds_per_s": rounds / (sk * 1e-3),
            "sweep_kernel_ms_reps": s_kern, "plain_kernel_ms_sum_reps": p_kern.tolist(),
            "parity": "checked %d of %d instances against the plain handles" % (checked, I)}


def reference_point(reps):
    seeds = np.arange(1, 65537, dtype=np.uint64)
    sim = BatchSimulator(seeds, 4, RandomDelay.new(10.0, 4.0)).create(1000)
    sim.run()
    k, w, res = timed(sim, reps)
    out = {"instances": 65536, "num_nodes": 4, "kernel": sim.kernel_info(), "kernel_ms": float(np.median(k)), "wall_ms": float(np.median(w)),
           "rounds_per_s": int(res.active_rounds.astype(np.int64).sum()) / (float(np.median(k)) * 1e-3), "kernel_ms_reps": k}
    sim.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True, check=True).stdout.strip()
    res = {"gpu": gpu, "reps": a.reps, "a_n4_64x1024": compare(4, 64, 1024, a.reps), "b_n7_16x1024": compare(7, 16, 1024, a.reps),
           "c_bench_65536x4": reference_point(a.reps)}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
