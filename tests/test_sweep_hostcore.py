"""Parameter sweeps (lbft_create_sweep) on the CPU: the sweep state machine (sim_core.cuh SW = true, compiled for the host by
tests/hostcore/sweepcore.cpp)
against the oracle run with each set's own plain configuration; the refusals of the product library; the ctypes layout of
lbft_param_set; the Python arguments."""
import ctypes
import os
import re

import numpy as np
import pytest

from librabft_simulator_b200 import _build, _lib
from librabft_simulator_b200._lib import LbftConfig, LbftParamSet
from tests import fuzz_configs
from tests.support import REF, Result, assert_same, make_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = ctypes.c_void_p
SET_KEYS = ("delay_kind", "delay_mean", "delay_variance", "delay_lo", "delay_hi", "target_commit_interval", "delta", "gamma",
            "lambda_", "silent")


def param_set(**kw):
    """lbft_param_set from oracle-style keywords (REF defaults; silent as a per-node list)."""
    s = LbftParamSet()
    s.struct_size = ctypes.sizeof(LbftParamSet)
    vals = dict(delay_kind=0, delay_lo=0, delay_hi=0, **{k: REF[k] for k in ("delay_mean", "delay_variance", "target_commit_interval",
                                                                              "delta", "gamma", "lambda_")})
    vals.update(kw)
    silent = vals.pop("silent", None)
    for k, v in vals.items():
        setattr(s, k, v)
    s.silent_mask = 0 if silent is None else sum(1 << i for i, f in enumerate(silent) if f)
    return s


@pytest.fixture(scope="module")
def sweepcore():
    lib = ctypes.CDLL(_build.build_sweepcore())
    lib.sweepcore_last_error.restype = ctypes.c_char_p
    lib.sweepcore_run.argtypes = [ctypes.POINTER(LbftConfig), ctypes.POINTER(LbftParamSet), ctypes.c_uint32, P, P, P, P, P, P, P]
    return lib


def run_sweep(sweepcore, seeds, num_nodes, max_clock, sets, set_of, **shared):
    cfg, keep = make_config(seeds, num_nodes, max_clock, **shared)
    arr = (LbftParamSet * len(sets))(*[param_set(**s) for s in sets])
    idx = np.ascontiguousarray(set_of, dtype=np.uint32)
    I = cfg.num_instances
    res = Result(I, num_nodes)
    res.lc_round = np.zeros((I, num_nodes), np.uint32)
    layout = np.zeros(4, np.uint32)
    rc = sweepcore.sweepcore_run(ctypes.byref(cfg), arr, len(sets), P(idx.ctypes.data), P(res.commit_counts.ctypes.data), P(res.last_states.ctypes.data),
            P(res.lc_round.ctypes.data), P(res.counters.ctypes.data), P(res.status.ctypes.data), P(layout.ctypes.data))
    if rc != 0:
        raise RuntimeError(sweepcore.sweepcore_last_error().decode())
    res.layout = dict(zip(("words", "queue_scan", "queue_cap", "payload_cap"), layout.tolist()))
    return res


def rows(res, sel):
    out = Result(int(sel.sum()), res.commit_counts.shape[1])
    out.commit_counts, out.last_states, out.counters, out.status = (res.commit_counts[sel], res.last_states[sel], res.counters[sel],
                                                                    res.status[sel])
    return out


def check_against_oracle(oracle, res, seeds, num_nodes, max_clock, sets, set_of, **shared):
    for k, s in enumerate(sets):
        sel = set_of == k
        if not sel.any():
            continue
        ref = oracle.run(seeds[sel], num_nodes, max_clock, **shared, **s)
        got = rows(res, sel)
        assert not (got.status & _lib.ST_ERROR_MASK).any(), "parameter set %d overflows its capacities: not a parity case" % k
        assert_same(got, ref, "(parameter set %d: %s)" % (k, s))
        np.testing.assert_array_equal(got.status, ref.status, err_msg="status differs (parameter set %d)" % k)


def interleaved(num_sets, per_set, seed):
    return np.random.default_rng(seed).permutation(np.arange(num_sets * per_set) % num_sets).astype(np.uint32)


SETS4 = [
    {},                                                        # the reference's defaults
    dict(delay_mean=5.0, delay_variance=1.0),
    dict(delay_mean=20.0, delay_variance=30.0),
    dict(delay_mean=10.0, delay_variance=0.0),                 # constant delay
    dict(delay_mean=3.0, delay_variance=0.0),
    dict(delay_mean=10.0, delay_variance=100.0),               # too wide for the threshold table: the exp() path
    dict(delay_kind=1, delay_lo=2, delay_hi=12),               # uniform
    dict(delay_kind=1, delay_lo=1, delay_hi=7),
    dict(delta=10, gamma=1.5, lambda_=1.0),
    dict(delta=40, gamma=1.0, lambda_=0.25, target_commit_interval=150),
    dict(target_commit_interval=1000, delay_mean=8.0, delay_variance=6.0),
    dict(silent=[0, 0, 0, 1]),
    dict(silent=[1, 0, 0, 0], delay_mean=7.0, delay_variance=3.0),
    dict(delay_mean=4.0, delay_variance=0.5, delta=15),
]
SETS7 = [
    {},
    dict(delay_mean=6.0, delay_variance=2.0, delta=30),
    dict(delay_kind=1, delay_lo=3, delay_hi=15),
    dict(silent=[0, 1, 0, 0, 0, 0, 1], gamma=1.5),
    dict(delay_mean=14.0, delay_variance=0.0, target_commit_interval=150),
]
PART7 = dict(partition_windows=4, partition_max_len=100)


def test_tables_cover_both_delay_paths(hostcore):
    assert hostcore.setup_info(4, **dict(REF))["delay_kmax"] > 0
    assert hostcore.setup_info(4, **dict(REF, delay_variance=100.0))["delay_kmax"] == 0


def test_sweep_of_four_author_sets_matches_the_oracle(sweepcore, oracle):
    set_of = interleaved(len(SETS4), 6, 1)
    seeds = np.arange(1000, 1000 + len(set_of), dtype=np.uint64)
    res = run_sweep(sweepcore, seeds, 4, 1000, SETS4, set_of)
    check_against_oracle(oracle, res, seeds, 4, 1000, SETS4, set_of)


def test_sweep_of_seven_authors_with_partitions_matches_the_oracle(sweepcore, oracle, monkeypatch):
    monkeypatch.setenv("LBFT_FORCE_KERNEL", "thread")   # the layout of the large-batch (thread-kernel) shape
    set_of = interleaved(len(SETS7), 5, 2)
    seeds = np.arange(77, 77 + len(set_of), dtype=np.uint64)
    res = run_sweep(sweepcore, seeds, 7, 1000, SETS7, set_of, **PART7)
    assert res.layout["queue_scan"] == 3   # calendar queue
    check_against_oracle(oracle, res, seeds, 7, 1000, SETS7, set_of, **PART7)


def test_sweep_on_the_heap_queue_matches_the_oracle(sweepcore, oracle):
    sets = [{}, dict(delay_mean=4.0, delay_variance=2.0), dict(delay_kind=1, delay_lo=5, delay_hi=25, delta=30)]
    set_of = interleaved(len(sets), 2, 3)
    seeds = np.arange(5, 5 + len(set_of), dtype=np.uint64)
    res = run_sweep(sweepcore, seeds, 6, 5000, sets, set_of)
    assert res.layout["queue_scan"] == 0   # binary heap (horizon beyond the calendar's)
    check_against_oracle(oracle, res, seeds, 6, 5000, sets, set_of)


def test_capacities_fit_the_fastest_set(hostcore, sweepcore, oracle):
    """A short mean delay raises the event rate past what the shared-memory queue's 16-bit stamps cover: the sweep takes the
    fast set's queue mode and every set's capacities, and each set still computes what its own plain handle computes."""
    slow, fast = {}, dict(delay_mean=1.0, delay_variance=0.25)
    plain = [hostcore.setup_info(4, 2000, **dict(REF, **s)) for s in (slow, fast)]
    assert plain[0]["queue_scan"] != plain[1]["queue_scan"]
    set_of = interleaved(2, 5, 4)
    seeds = np.arange(300, 310, dtype=np.uint64)
    res = run_sweep(sweepcore, seeds, 4, 2000, [slow, fast], set_of)
    assert res.layout["queue_scan"] == plain[1]["queue_scan"]
    assert res.layout["queue_cap"] >= max(p["queue_cap"] for p in plain)
    assert res.layout["payload_cap"] >= max(p["payload_cap"] for p in plain)
    check_against_oracle(oracle, res, seeds, 4, 2000, [slow, fast], set_of)


def test_one_set_sweep_equals_the_plain_host_core(hostcore, sweepcore):
    rng = np.random.default_rng(2024)
    done = 0
    while done < 6:
        n, max_clock, seed0, kw = fuzz_configs.random_config(rng)
        if "commands_per_epoch" in kw:
            continue   # sweeps are single-epoch
        seeds = np.arange(seed0, seed0 + 8, dtype=np.uint64)
        plain = hostcore.run(seeds, n, max_clock, **kw)
        shared = {k: v for k, v in kw.items() if k not in SET_KEYS}
        s = {k: v for k, v in kw.items() if k in SET_KEYS}
        res = run_sweep(sweepcore, seeds, n, max_clock, [s], np.zeros(8, np.uint32), **shared)
        for f in ("commit_counts", "last_states", "lc_round", "counters", "status"):
            np.testing.assert_array_equal(getattr(res, f), getattr(plain, f), err_msg="%s (N=%d, %s)" % (f, n, kw))
        assert res.layout["words"] == plain.words_per_instance
        done += 1


# ---- the product library: refusals before the device check ------------------------------------------------------------

@pytest.fixture(scope="module")
def lib():
    _build.build_product()
    return _lib.load()


def create_sweep(lib, sets, set_of, num_sets=None, seeds=(1, 2, 3, 4), **cfg_kw):
    cfg, keep = make_config(list(seeds), 4, **cfg_kw)
    arr = (LbftParamSet * max(1, len(sets)))(*[param_set(**s) for s in sets])
    idx = np.ascontiguousarray(set_of, dtype=np.uint32)
    h = ctypes.c_void_p()
    rc = lib.lbft_create_sweep(ctypes.byref(cfg), arr, len(sets) if num_sets is None else num_sets, P(idx.ctypes.data), ctypes.byref(h))
    if rc == 0:
        lib.lbft_destroy(h)
    return rc, lib.lbft_last_error().decode()


@pytest.mark.parametrize("case, expect", [
    (dict(flags=1), "flags must be 0"),
    (dict(flags=2), "flags must be 0"),
    (dict(commands_per_epoch=10), "commands_per_epoch >= round_cap"),
    (dict(num_sets=0), "num_sets"),
    (dict(num_sets=_lib.MAX_PARAM_SETS + 1), "num_sets"),
    (dict(set_of=[0, 1, 2, 0]), "set_of_instance[2] = 2 is out of range"),
    (dict(sets=[{}, dict(delta=0)]), "parameter set 1: delta = 0"),
    (dict(sets=[{}, dict(delay_mean=-1.0)]), "parameter set 1: LogNormal delay needs mean > 0"),
    (dict(sets=[{}, dict(delay_variance=-1.0)]), "parameter set 1: LogNormal delay needs mean > 0 and variance >= 0"),
    (dict(sets=[dict(delay_kind=1, delay_lo=5, delay_hi=2), {}]), "parameter set 0: uniform delay"),
    (dict(sets=[{}, dict(delay_mean=1e12, delay_variance=0.0)]), "parameter set 1: constant delay out of range"),
    (dict(sets=[{}, dict(silent=[0, 0, 0, 0, 1])]), "parameter set 1: silent_mask has bits at or above num_nodes"),
    (dict(sets=[{}, dict(delay_kind=5)]), "parameter set 1: unknown delay_kind"),
])
def test_invalid_sweeps_are_refused(lib, case, expect):
    case = dict(case)
    sets = case.pop("sets", [{}, {}])
    set_of = case.pop("set_of", [0, 1, 0, 1])
    num_sets = case.pop("num_sets", None)
    if num_sets == 0:
        sets = []
    elif num_sets is not None:
        sets = [{}] * num_sets
    rc, msg = create_sweep(lib, sets, set_of, num_sets=num_sets, **case)
    assert rc == -1, (case, msg)
    assert expect in msg


def test_a_set_with_the_wrong_struct_size_is_refused(lib):
    cfg, keep = make_config([1, 2], 4)
    arr = (LbftParamSet * 1)(param_set())
    arr[0].struct_size = 8
    idx = np.zeros(2, np.uint32)
    h = ctypes.c_void_p()
    assert lib.lbft_create_sweep(ctypes.byref(cfg), arr, 1, P(idx.ctypes.data), ctypes.byref(h)) == -1
    assert b"struct_size" in lib.lbft_last_error()
    assert lib.lbft_create_sweep(ctypes.byref(cfg), None, 1, P(idx.ctypes.data), ctypes.byref(h)) == -1
    assert lib.lbft_create_sweep(ctypes.byref(cfg), arr, 1, None, ctypes.byref(h)) == -1


def test_a_valid_sweep_has_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    rc, msg = create_sweep(lib, [{}, dict(delay_mean=5.0)], [0, 1, 1, 0])
    assert rc == -2 and "no CPU fallback" in msg


def test_param_set_layout_matches_the_header():
    header = open(os.path.join(ROOT, "include", "lbft.h")).read()
    body = re.search(r"typedef struct lbft_param_set \{(.*?)\} lbft_param_set;", re.sub(r"/\*.*?\*/", "", header, flags=re.S), re.S).group(1)
    ctype = {"uint32_t": ctypes.c_uint32, "int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64, "double": ctypes.c_double}
    fields = []
    for decl in [d.strip() for d in body.split(";") if d.strip()]:
        t, names = decl.split(None, 1)
        fields += [(n.strip(), ctype[t]) for n in names.split(",")]
    got = [("lambda" if n == "lambda_" else n, t) for n, t in LbftParamSet._fields_]
    assert got == fields
    assert ctypes.sizeof(LbftParamSet) == 80
    assert int(re.search(r"#define LBFT_MAX_PARAM_SETS (\d+)u", header).group(1)) == _lib.MAX_PARAM_SETS >= 1024


# ---- Python mirror -------------------------------------------------------------------------------------------------

def test_python_sweep_arguments(lib):
    from librabft_simulator_b200 import BatchSimulator, NodeConfig, ParamSet, RandomDelay
    sets = [ParamSet(), ParamSet(RandomDelay.uniform(2, 9), NodeConfig(delta=30), silent=[0, 1, 0, 0]), ParamSet(RandomDelay.new(5.0, 1.0))]
    sim = BatchSimulator(np.arange(1, 8), 4, param_sets=sets)
    np.testing.assert_array_equal(sim.set_index, np.arange(7) % 3)
    assert sim.set_index.dtype == np.uint32
    c = sets[1].to_c()
    assert (c.delay_kind, c.delay_lo, c.delay_hi, c.delta, c.silent_mask) == (1, 2, 9, 30, 2)
    assert c.struct_size == ctypes.sizeof(LbftParamSet)
    sim = BatchSimulator(np.arange(1, 5), 4, param_sets=sets, set_index=[2, 2, 0, 1])
    np.testing.assert_array_equal(sim.set_index, [2, 2, 0, 1])
    for bad in (dict(network_delay=RandomDelay.new(5.0, 1.0)), dict(node_config=NodeConfig(delta=5)), dict(silent=[0, 0, 0, 1])):
        with pytest.raises(ValueError, match="param_sets"):
            BatchSimulator(np.arange(1, 5), 4, param_sets=sets, **bad)
    with pytest.raises(ValueError, match="one entry per seed"):
        BatchSimulator(np.arange(1, 5), 4, param_sets=sets, set_index=[0, 1])
    with pytest.raises(ValueError, match="needs param_sets"):
        BatchSimulator(np.arange(1, 5), 4, set_index=[0, 0, 0, 0])
    with pytest.raises(ValueError, match="non-empty"):
        BatchSimulator(np.arange(1, 5), 4, param_sets=[])
