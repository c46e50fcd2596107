"""bench.py --dump-outputs (host side, no GPU): what it writes for a batch result, and that the benchmark's own build of
the CPU baseline stays out of the source tree."""
import os
import subprocess
import sys
import types

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fake_result(instances, nodes, seed=7):
    rng = np.random.default_rng(seed)
    return types.SimpleNamespace(
        commit_counts=rng.integers(0, 2 ** 32, (instances, nodes), dtype=np.uint64).astype(np.uint32),
        last_committed_states=rng.integers(0, 2 ** 64, (instances, nodes), dtype=np.uint64),
        active_rounds=rng.integers(0, 2 ** 32, instances, dtype=np.uint64).astype(np.uint32),
        status=np.full(instances, 1, np.uint32),
        counters=rng.integers(0, 2 ** 32, (instances, 12), dtype=np.uint64).astype(np.uint32))


def load(out):
    return {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}


def test_dump_is_float64_and_loses_nothing(tmp_path):
    res = fake_result(100, 5)
    bench.dump_outputs(res, str(tmp_path))
    got = load(str(tmp_path))
    assert sorted(got) == ["active_rounds", "commit_counts", "counters", "instance", "last_committed_states_hi",
                           "last_committed_states_lo", "status"]
    assert all(a.dtype == np.float64 for a in got.values())
    np.testing.assert_array_equal(got["instance"], np.arange(100))
    states = (got["last_committed_states_hi"].astype(np.uint64) << np.uint64(32)) | got["last_committed_states_lo"].astype(np.uint64)
    np.testing.assert_array_equal(states, res.last_committed_states)
    for name in ("commit_counts", "active_rounds", "status", "counters"):
        np.testing.assert_array_equal(got[name].astype(np.uint64), getattr(res, name))


def test_large_dump_is_a_fixed_sample_within_the_limit(tmp_path):
    res = fake_result(5000, 8)
    limit = 200_000
    for run in ("a", "b"):
        bench.dump_outputs(res, str(tmp_path / run), limit_bytes=limit)
    a, b = load(str(tmp_path / "a")), load(str(tmp_path / "b"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= limit
    rows = a["instance"].astype(np.int64)
    assert 0 < len(rows) < 5000 and (np.diff(rows) > 0).all()
    for name in a:
        np.testing.assert_array_equal(a[name], b[name])
    np.testing.assert_array_equal(a["commit_counts"], res.commit_counts[rows])
    np.testing.assert_array_equal(a["counters"], res.counters[rows])


def test_native_oracle_is_private_to_its_process_and_outside_the_tree():
    """The -O3 -march=native oracle is compiled into a fresh directory only its user can write, outside the source tree,
    and the directory is gone once the process that built it exits (no shared cache another user could plant a library in)."""
    code = ("import os, sys; sys.path.insert(0, %r); from librabft_simulator_b200 import _build; "
            "p, f = _build.build_oracle_native(); assert _build.build_oracle_native() == (p, f); st = os.lstat(os.path.dirname(p)); "
            "print(p, f, st.st_uid, oct(st.st_mode & 0o7777), sep='|')" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, text=True, check=True).stdout
    path, flags, uid, mode = out.strip().splitlines()[-1].split("|")
    assert flags == "-O3 -march=native"
    assert not os.path.abspath(path).startswith(ROOT + os.sep), path
    assert int(uid) == os.getuid() and mode == "0o700", (uid, mode)
    assert not os.path.exists(os.path.dirname(path)), path
