"""Parameter sweeps on the B200: every instance of a sweep handle equals the oracle run with its own set's plain
configuration, on both kernel families, through every read-out path (summaries, commit logs, run_stream, plain C)."""
import os
import subprocess

import numpy as np
import pytest

from librabft_simulator_b200 import BatchSimulator, NodeConfig, ParamSet, RandomDelay
from tests.support import REF, Result, assert_same
from tests.test_gpu_cabi_c import build_c_caller
from tests.test_sweep_hostcore import PART7, SETS4, SETS7, interleaved


def to_param_set(d):
    v = dict(REF, delay_kind=0, delay_lo=0, delay_hi=0)
    v.update(d)
    delay = RandomDelay.uniform(v["delay_lo"], v["delay_hi"]) if v["delay_kind"] == 1 else RandomDelay.new(v["delay_mean"], v["delay_variance"])
    return ParamSet(delay, NodeConfig(v["target_commit_interval"], v["delta"], v["gamma"], v["lambda_"]), v.get("silent"))


def as_result(res, sel):
    out = Result(int(sel.sum()), res.commit_counts.shape[1])
    out.commit_counts, out.last_states = res.commit_counts[sel], res.last_committed_states[sel]
    out.counters, out.status = res.counters[sel], res.status[sel]
    return out


def check_sets(oracle, res, seeds, num_nodes, max_clock, sets, **shared):
    assert res.set_index is not None
    for k, s in enumerate(sets):
        sel = res.set_index == k
        if not sel.any():
            continue
        ref = oracle.run(seeds[sel], num_nodes, max_clock, **shared, **s)
        got = as_result(res, sel)
        assert_same(got, ref, "(parameter set %d: %s)" % (k, s))
        np.testing.assert_array_equal(got.status, ref.status, err_msg="status differs (parameter set %d)" % k)
        np.testing.assert_array_equal(res.active_rounds[sel], ref.counters[:, 6], err_msg="active rounds (parameter set %d)" % k)


def run_sweep(seeds, num_nodes, max_clock, sets, set_of, **shared):
    sim = BatchSimulator(seeds, num_nodes, param_sets=[to_param_set(s) for s in sets], set_index=set_of, **shared)
    res = sim.loop_until(max_clock)
    return sim, res


SETS64 = [{}, dict(delay_mean=6.0, delay_variance=2.0, delta=30), dict(silent=[1] * 5 + [0] * 59, gamma=1.5)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["n4", "n7_partitions", "n64"])
def test_sweep_matches_the_oracle_per_set(oracle, kernel_choice, shape):
    if shape == "n4":
        N, clock, sets, shared, per = 4, 1000, SETS4, {}, 8
    elif shape == "n7_partitions":
        N, clock, sets, shared, per = 7, 1000, SETS7, PART7, 8
    else:
        N, clock, sets, shared, per = 64, 1000, SETS64, {}, 2
    set_of = interleaved(len(sets), per, 11)
    seeds = np.arange(9000, 9000 + len(set_of), dtype=np.uint64)
    sim, res = run_sweep(seeds, N, clock, sets, set_of, **shared)
    want = "lbft_sweep_wide_kernel<" if kernel_choice == "wide" else "lbft_sweep_kernel<"
    assert sim.kernel_info().startswith(want), sim.kernel_info()
    check_sets(oracle, res, seeds, N, clock, sets, **shared)
    sim.close()


def grid_sets(n):
    """A Monte-Carlo grid over the knobs the reference exposes: mean / variance of the delay, delta, gamma, lambda, plus uniform
    delays and a silent node."""
    out = []
    for k in range(n):
        s = dict(delay_mean=6.0 + 2.0 * (k % 8), delay_variance=[0.0, 1.0, 4.0, 9.0][(k // 8) % 4], delta=[15, 20, 30, 40][k % 4],
                 gamma=[1.5, 2.0][(k // 2) % 2], lambda_=[0.5, 1.0][(k // 16) % 2])
        if k % 13 == 5:
            s = dict(delay_kind=1, delay_lo=3 + k % 4, delay_hi=12 + k % 7, delta=s["delta"])
        if k % 11 == 3:
            s["silent"] = [0, 0, 0, 1]
        out.append(s)
    return out


@pytest.mark.gpu
def test_sixty_four_sets_of_1024_seeds_match_the_oracle(oracle):
    sets = grid_sets(64)
    set_of = interleaved(64, 1024, 12)
    seeds = np.arange(1, 65537, dtype=np.uint64)
    sim, res = run_sweep(seeds, 4, 1000, sets, set_of)
    assert not (res.status & 0x9e).any()
    check_sets(oracle, res, seeds, 4, 1000, sets)
    sim.close()


@pytest.mark.gpu
def test_sweep_commit_logs_match_the_oracle(oracle, kernel_choice):
    set_of = interleaved(len(SETS4), 3, 13)
    seeds = np.arange(40, 40 + len(set_of), dtype=np.uint64)
    sim, res = run_sweep(seeds, 4, 1000, SETS4, set_of)
    rows, lens = res.commit_logs()
    for i in range(len(seeds)):
        s = SETS4[set_of[i]]
        for node in range(4):
            want = oracle.commit_log([seeds[i]], 4, 0, node, 1000, **s)
            got = [(int(r["proposer"]), int(r["index"]), int(r["time"])) for r in rows[i, :lens[i, node]]]
            assert got == want, (i, node, s)
    sim.close()


@pytest.mark.gpu
def test_run_stream_on_a_sweep_handle(oracle):
    sets = SETS4[:6]
    set_of = interleaved(len(sets), 40, 14)
    batches = [np.arange(b * 1000, b * 1000 + len(set_of), dtype=np.uint64) for b in range(3)]
    sim = BatchSimulator(batches[0], 4, param_sets=[to_param_set(s) for s in sets], set_index=set_of).create(1000)
    n = 0
    for seeds, res in zip(batches, sim.run_stream(batches)):
        np.testing.assert_array_equal(res.set_index, set_of)
        check_sets(oracle, res, seeds, 4, 1000, sets)
        n += 1
    assert n == 3
    sim.close()


def test_c_sweep_caller_compiles_and_links(tmp_path):
    assert os.path.exists(build_c_caller(tmp_path, "sweep_run"))


@pytest.mark.gpu
def test_c_sweep_caller_matches_the_oracle(tmp_path, oracle):
    exe = build_c_caller(tmp_path, "sweep_run")
    p = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert p.returncode == 0, p.stdout
    assert "sweep ok" in p.stdout
    sets = [{}, dict(delay_kind=1, delay_lo=2, delay_hi=12), dict(silent=[0, 0, 0, 1], delta=30)]
    lines = [ln.split() for ln in p.stdout.splitlines() if ln.startswith("inst ")]
    assert len(lines) == 96
    for ln in lines:
        i, k = int(ln[1]), int(ln[2])
        ref = oracle.run([500 + i], 4, 1000, **sets[k])
        assert [int(v) for v in ln[3:7]] == ref.commit_counts[0].tolist(), ln
        assert [int(v) for v in ln[7:11]] == ref.last_states[0].tolist(), ln
