"""Host-side mirror of the reference's simulator interface over the C ABI.

Reference surface being mirrored (novifinancial/librabft_simulator):

* ``bft_lib::simulator::RandomDelay::new(mean, variance)``                     simulator.rs:99-106
* ``librabft_v2::node::NodeConfig {target_commit_interval, delta, gamma, lambda}``  node.rs:76-81
* ``bft_lib::simulator::Simulator::new(seed, num_nodes, delay, context_factory)``   simulator.rs:200-208
* ``Simulator::loop_until(GlobalTime(max_clock), csv_path) -> Vec<&Context>``       simulator.rs:380
* ``SimulatedContext::committed_history()`` / ``last_committed_state()``            simulated_context.rs:98-100,194-196

``BatchSimulator`` is the batched form (one handle = many independent ``Simulator`` instances, one per seed,
advanced in lockstep on one B200); ``Simulator`` is the single-instance spelling of the reference.  All the
simulation work happens in the CUDA library; this module only marshals arguments and results.
"""
import ctypes
import os
from dataclasses import dataclass

import numpy as np

from . import _lib

DELAY_LOGNORMAL, DELAY_UNIFORM = 0, 1
# one row of committed_history(): include/lbft.h lbft_commit
COMMIT_DTYPE = np.dtype([("proposer", np.uint32), ("index", np.uint32), ("time", np.int64)])


@dataclass(frozen=True)
class RandomDelay:
    """``RandomDelay`` (simulator.rs:39-43).  ``new`` is the reference's LogNormal; ``uniform`` is an extension."""
    kind: int = DELAY_LOGNORMAL
    mean: float = 10.0
    variance: float = 4.0
    lo: int = 0
    hi: int = 0

    @staticmethod
    def new(mean, variance):
        return RandomDelay(DELAY_LOGNORMAL, float(mean), float(variance))

    @staticmethod
    def uniform(lo, hi):
        return RandomDelay(DELAY_UNIFORM, 0.0, 0.0, int(lo), int(hi))


@dataclass(frozen=True)
class NodeConfig:
    """``NodeConfig`` (node.rs:76-81) with the CLI defaults of main.rs:72-172."""
    target_commit_interval: int = 100000
    delta: int = 20
    gamma: float = 2.0
    lambda_: float = 0.5


@dataclass(frozen=True)
class ParamSet:
    """One parameter set of a sweep: the knobs a Monte-Carlo study moves (network delay, pacemaker ``NodeConfig``, silent
    nodes).  ``silent`` is ``None`` or a per-node sequence of flags, like ``BatchSimulator(silent=...)``."""
    network_delay: RandomDelay = RandomDelay()
    node_config: NodeConfig = NodeConfig()
    silent: tuple = None

    def to_c(self):
        s = _lib.LbftParamSet()
        s.struct_size = ctypes.sizeof(_lib.LbftParamSet)
        d, n = self.network_delay, self.node_config
        s.delay_kind, s.delay_mean, s.delay_variance, s.delay_lo, s.delay_hi = d.kind, d.mean, d.variance, d.lo, d.hi
        s.target_commit_interval, s.delta, s.gamma, s.lambda_ = n.target_commit_interval, n.delta, n.gamma, n.lambda_
        s.silent_mask = 0 if self.silent is None else sum(1 << i for i, f in enumerate(self.silent) if f)
        return s


@dataclass(frozen=True)
class GlobalTime:
    """``GlobalTime(i64)`` (simulator.rs:35-37)."""
    value: int

    def __int__(self):
        return int(self.value)


@dataclass(frozen=True)
class Command:
    """``Command {proposer, index}`` (simulated_context.rs:31-35)."""
    proposer: int
    index: int


class SimulatedContextView:
    """Read-only view of one node's ``SimulatedContext`` after the run (simulated_context.rs:74-100)."""

    def __init__(self, batch, instance, author):
        self._batch, self._instance, self.author = batch, instance, author

    def committed_history(self):
        """``committed_history()`` -> list of ``(Command, NodeTime)`` (simulated_context.rs:98-100)."""
        return [(Command(p, i), t) for (p, i, t) in self._batch.commit_log(self._instance, self.author)]

    def last_committed_state(self):
        """``StateFinalizer::last_committed_state()`` -> the ``State(u64)`` key (simulated_context.rs:194-196)."""
        return int(self._batch.last_committed_states[self._instance, self.author])

    def num_commits(self):
        return int(self._batch.commit_counts[self._instance, self.author])


class BatchResult:
    """Results of ``BatchSimulator.loop_until``: what the reference's callers read from ``Vec<&Context>``.

    The summary arrays (commit counts, state keys, status, rounds) are copied out of the library's pinned result
    buffers when the result is created, so a ``BatchResult`` keeps describing ITS run after the handle has been
    re-run, re-seeded or closed.  Counters and commit logs are read on demand and are only available until the
    handle runs again (a stale read raises instead of returning another run's data)."""

    def __init__(self, sim):
        self._sim = sim
        self._generation = sim._generation
        I, N = sim.num_instances, sim.num_nodes
        #: ``committed_history().len()`` per node: [instance, node]
        self.commit_counts = sim._fetch("lbft_commit_counts", np.uint32, (I, N))
        #: ``last_committed_state()`` per node (SipHash-1-3 key of the commit log): [instance, node]
        self.last_committed_states = sim._fetch("lbft_last_states", np.uint64, (I, N))
        #: max over nodes of ``ActiveRound::active_round()`` per instance (simulator.rs:86-88)
        self.active_rounds = sim._fetch("lbft_active_rounds", np.uint32, (I,))
        self.status = sim._fetch("lbft_status", np.uint32, (I,))
        #: parameter set of each instance (sweeps; ``None`` for a plain batch)
        self.set_index = None if sim.set_index is None else sim.set_index.copy()
        self._counters = None

    @property
    def counters(self):
        """lbft_instance_counters per instance, [instance, 12] (fetched on first use; 48 bytes per instance)."""
        if self._counters is None:
            self._check_current("counters")
            self._counters = self._sim._fetch("lbft_counters", np.uint32, (self._sim.num_instances, 12))
        return self._counters

    def _check_current(self, what):
        if self._sim._handle is None or self._generation != self._sim._generation:
            raise RuntimeError("the %s of this result are gone: the simulator has been run again (or closed) since; read "
                               "them before the next run" % what)

    # lbft_instance_counters columns
    @property
    def events_processed(self):
        return self.counters[:, 0:4].sum(axis=1)

    def commit_log(self, instance, author):
        self._check_current("commit logs")
        return self._sim.commit_log(instance, author)

    def commit_logs(self, cap=None):
        """All commit logs of the batch in one device pass (``lbft_commit_logs``): ``(rows[instance, cap], lens[instance,
        node])``; node n's ``committed_history()`` is ``rows[instance, :lens[instance, n]]``."""
        self._check_current("commit logs")
        return self._sim.commit_logs(cap)

    def contexts(self, instance=0):
        """The ``Vec<&Context>`` that ``loop_until`` returns for one instance."""
        return [SimulatedContextView(self, instance, a) for a in range(self._sim.num_nodes)]


class BatchSimulator:
    """Many independent ``Simulator`` instances (one per seed) on one GPU.

    ``param_sets`` (a sequence of ``ParamSet``) makes the batch a parameter sweep: instance i runs with
    ``param_sets[set_index[i]]`` instead of ``network_delay`` / ``node_config`` / ``silent`` (which must then keep their
    defaults) and computes exactly what a plain batch with that set would compute for its seed.  ``set_index`` defaults to
    ``arange(num_instances) % len(param_sets)``."""

    def __init__(self, seeds, num_nodes, network_delay=RandomDelay(), node_config=NodeConfig(),
                 commands_per_epoch=30000, voting_rights=None, silent=None, partition_windows=0,
                 partition_max_len=0, device=0, round_cap=0, queue_cap=0, payload_cap=0, record_round_switches=False, resumable=False,
                 true_data_sync=False, param_sets=None, set_index=None):
        self._lib = _lib.load()
        self.record_round_switches = bool(record_round_switches)  # LBFT_FLAG_ROUND_SWITCHES (DataWriter, data_writer.rs)
        self.resumable = bool(resumable)  # LBFT_FLAG_RESUMABLE: run_until / snapshot / restore
        # LBFT_FLAG_TRUE_DATA_SYNC: NON-PARITY variant — requests are answered by the node they were sent to (the reference
        # simulator dispatches them to the requester itself, simulator.rs:446)
        self.true_data_sync = bool(true_data_sync)
        self.seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64).reshape(-1))
        self.num_instances = int(self.seeds.shape[0])
        self.num_nodes = int(num_nodes)
        self.network_delay, self.node_config = network_delay, node_config
        self.commands_per_epoch = int(commands_per_epoch)
        self.voting_rights = None if voting_rights is None else np.ascontiguousarray(voting_rights, dtype=np.uint64)
        self.silent = None if silent is None else np.ascontiguousarray(silent, dtype=np.uint8)
        self.partition_windows, self.partition_max_len = int(partition_windows), int(partition_max_len)
        self.device, self.round_cap, self.queue_cap, self.payload_cap = int(device), int(round_cap), int(queue_cap), int(payload_cap)
        self.param_sets, self.set_index = None, None
        if param_sets is not None:
            if network_delay != RandomDelay() or node_config != NodeConfig() or silent is not None:
                raise ValueError("network_delay, node_config and silent come from param_sets in a sweep: leave them at their defaults")
            self.param_sets = list(param_sets)
            if not self.param_sets or any(not isinstance(p, ParamSet) for p in self.param_sets):
                raise ValueError("param_sets must be a non-empty sequence of ParamSet")
            idx = np.arange(self.num_instances) % len(self.param_sets) if set_index is None else set_index
            self.set_index = np.ascontiguousarray(np.asarray(idx).reshape(-1), dtype=np.uint32)
            if self.set_index.shape[0] != self.num_instances:
                raise ValueError("set_index needs one entry per seed (%d)" % self.num_instances)
        elif set_index is not None:
            raise ValueError("set_index needs param_sets")
        self._handle = None
        self._generation = 0   # bumped by every run: results of an older run know they are stale
        self.timing = None

    # -- lifetime -------------------------------------------------------------------------------
    def make_config(self, max_clock):
        c = _lib.LbftConfig()
        c.struct_size = ctypes.sizeof(_lib.LbftConfig)
        c.num_instances, c.num_nodes = self.num_instances, self.num_nodes
        c.delay_kind = self.network_delay.kind
        c.seeds = self.seeds.ctypes.data
        c.max_clock = int(max_clock)
        c.delay_mean, c.delay_variance = self.network_delay.mean, self.network_delay.variance
        c.delay_lo, c.delay_hi = self.network_delay.lo, self.network_delay.hi
        c.target_commit_interval, c.delta = self.node_config.target_commit_interval, self.node_config.delta
        c.gamma, c.lambda_ = self.node_config.gamma, self.node_config.lambda_
        c.commands_per_epoch = self.commands_per_epoch
        c.voting_rights = None if self.voting_rights is None else self.voting_rights.ctypes.data
        c.silent = None if self.silent is None else self.silent.ctypes.data
        c.partition_windows, c.partition_max_len = self.partition_windows, self.partition_max_len
        c.device, c.round_cap, c.queue_cap, c.payload_cap = self.device, self.round_cap, self.queue_cap, self.payload_cap
        c.flags = ((_lib.FLAG_ROUND_SWITCHES if self.record_round_switches else 0) | (_lib.FLAG_RESUMABLE if self.resumable else 0) |
                   (_lib.FLAG_TRUE_DATA_SYNC if self.true_data_sync else 0))
        return c

    def create(self, max_clock):
        """``lbft_create``: validate, build the host tables, allocate device state."""
        self.close()
        handle = ctypes.c_void_p()
        cfg = self.make_config(max_clock)
        if self.param_sets is None:
            _lib.check(self._lib.lbft_create(ctypes.byref(cfg), ctypes.byref(handle)))
        else:
            sets = (_lib.LbftParamSet * len(self.param_sets))(*[p.to_c() for p in self.param_sets])
            _lib.check(self._lib.lbft_create_sweep(ctypes.byref(cfg), sets, len(self.param_sets),
                                                   ctypes.c_void_p(self.set_index.ctypes.data), ctypes.byref(handle)))
        self._handle = handle
        return self

    def close(self):
        if self._handle is not None:
            self._lib.lbft_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- running --------------------------------------------------------------------------------
    def loop_until(self, max_clock, csv_path=None, strict=True):
        """``Simulator::new`` + ``loop_until(max_clock)`` for every instance; host buffers in, host results out."""
        if csv_path is not None:
            # simulator.rs:380-381, 470-472: a DataWriter is kept during the loop and written at the end
            if self.num_instances != 1:
                raise ValueError("csv_path names ONE simulator's output directory: for a batch pass record_round_switches=True "
                                 "and call write_data_files(path, instance)")
            self.record_round_switches = True
        self.create(int(max_clock))
        self._generation += 1
        code = self._lib.lbft_run(self._handle)
        _lib.check(code, allow=() if strict else (_lib.LBFT_ERR_CAPACITY,))
        self._read_timing()
        if csv_path is not None:
            self.write_data_files(csv_path, 0)
        return BatchResult(self)

    def run_until(self, stop_clock, strict=True):
        """``lbft_run_until``: ``loop_until(GlobalTime(stop_clock), ..)`` on every instance of a resumable handle created
        with the final horizon (``create(horizon)``); the first call is ``Simulator::new`` + ``loop_until``, later calls
        continue — and, like the reference, each call drops the first event beyond its clock (simulator.rs:383-391)."""
        self._generation += 1
        code = self._lib.lbft_run_until(self._handle, int(stop_clock))
        _lib.check(code, allow=() if strict else (_lib.LBFT_ERR_CAPACITY,))
        self._read_timing()
        return BatchResult(self)

    def snapshot(self):
        """``lbft_snapshot_save``: the whole batch between two ``run_until`` calls, as a ``numpy.uint8`` array."""
        n = ctypes.c_size_t(0)
        _lib.check(self._lib.lbft_snapshot_size(self._handle, ctypes.byref(n)))
        buf = np.empty(n.value, dtype=np.uint8)
        _lib.check(self._lib.lbft_snapshot_save(self._handle, ctypes.c_void_p(buf.ctypes.data), n.value))
        return buf

    def restore(self, snapshot):
        """``lbft_snapshot_load`` into a handle created from the same configuration; continue with ``run_until``."""
        buf = np.ascontiguousarray(snapshot, dtype=np.uint8)
        self._generation += 1
        _lib.check(self._lib.lbft_snapshot_load(self._handle, ctypes.c_void_p(buf.ctypes.data), buf.nbytes))

    def set_seeds(self, seeds):
        """Re-seed the batch: the next run is a fresh ``Simulator::new(seed, ..)`` per instance."""
        seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64).reshape(-1))
        if seeds.shape[0] != self.num_instances:
            raise ValueError("expected %d seeds" % self.num_instances)
        self.seeds = seeds
        _lib.check(self._lib.lbft_set_seeds(self._handle, ctypes.c_void_p(seeds.ctypes.data)))

    def run(self, strict=True):
        """``lbft_run`` on the existing handle: seeds host->device, event-loop kernel, summaries device->host."""
        self._generation += 1
        code = self._lib.lbft_run(self._handle)
        _lib.check(code, allow=() if strict else (_lib.LBFT_ERR_CAPACITY,))
        self._read_timing()
        return BatchResult(self)

    def run_async(self):
        """``lbft_run_async``: enqueue upload + kernel + download on the handle's stream and return at once; the previous
        run's ``BatchResult`` stays valid, and ``set_seeds`` may stage the next batch meanwhile.  Finish with ``wait()``."""
        _lib.check(self._lib.lbft_run_async(self._handle))

    def wait(self, strict=True, relaunch=False, before_relaunch=None):
        """``lbft_wait``: block until the run started by ``run_async`` is done; returns its ``BatchResult``.

        ``relaunch=True`` starts the next run (``lbft_run_async`` on the seeds staged by ``set_seeds`` meanwhile) BEFORE the
        finished run's summaries are copied out of the pinned mirrors, so that the host-side copies overlap the next
        kernel: the library keeps two sets of mirrors and the getters serve the finished run while the next one is in
        flight.  ``before_relaunch()`` runs between the two (the multi-GPU all-gather reads the device buffers there)."""
        self._generation += 1
        code = self._lib.lbft_wait(self._handle)
        _lib.check(code, allow=() if strict else (_lib.LBFT_ERR_CAPACITY,))
        self._read_timing()
        if before_relaunch is not None:
            before_relaunch()
        if relaunch:
            self.run_async()
        return BatchResult(self)

    def run_stream(self, batches, strict=True):
        """Run a sequence of seed batches with one run always in flight: yields one ``BatchResult`` per batch, in order.
        Batch k + 1 is staged (pinned seed buffer) while batch k runs and launched the moment batch k's results have
        landed; each step still copies its seeds host->device and its summaries device->host."""
        it = iter(batches)
        first = next(it, None)
        if first is None:
            return
        self.set_seeds(first)
        self.run_async()
        inflight = True
        try:
            for nxt in it:
                self.set_seeds(nxt)
                inflight = False
                res = self.wait(strict=strict, relaunch=True)
                inflight = True
                yield res
            inflight = False
            yield self.wait(strict=strict)
        finally:
            if inflight:  # the consumer stopped early (or a batch failed to stage): drain the run that is still in flight
                self.drain()

    def drain(self):
        """Wait for an in-flight ``run_async`` and discard its result, leaving the handle idle (no-op if there is none)."""
        if self._handle is not None and self._lib.lbft_wait(self._handle) == _lib.LBFT_OK:
            self._generation += 1

    def device_buffer(self, which):
        """(device pointer, bytes) of a result buffer: 0 commit counts, 1 last states, 2 counters, 3 status."""
        ptr, nbytes = ctypes.c_void_p(), ctypes.c_size_t()
        _lib.check(self._lib.lbft_device_buffer(self._handle, which, ctypes.byref(ptr), ctypes.byref(nbytes)))
        return int(ptr.value), int(nbytes.value)

    def upload(self):
        _lib.check(self._lib.lbft_upload(self._handle))

    def run_device(self):
        self._generation += 1
        _lib.check(self._lib.lbft_run_device(self._handle))
        self._read_timing()

    def download(self, strict=True):
        _lib.check(self._lib.lbft_download(self._handle), allow=() if strict else (_lib.LBFT_ERR_CAPACITY,))
        self._read_timing()
        return BatchResult(self)

    def _read_timing(self):
        t = _lib.LbftTiming()
        _lib.check(self._lib.lbft_timing_info(self._handle, ctypes.byref(t)))
        self.timing = t

    def kernel_info(self):
        """Name of the kernel instantiation the handle launches (as ncu / cuobjdump spell it)."""
        buf = ctypes.create_string_buffer(128)
        _lib.check(self._lib.lbft_kernel_info(self._handle, buf, 128))
        return buf.value.decode()

    def memory_info(self):
        b, w = ctypes.c_uint64(), ctypes.c_uint32()
        _lib.check(self._lib.lbft_memory_info(self._handle, ctypes.byref(b), ctypes.byref(w)))
        return int(b.value), int(w.value)

    # -- results --------------------------------------------------------------------------------
    def _fetch(self, fn, dtype, shape):
        if self._handle is None:
            raise RuntimeError("the simulator has been closed (or not created): results are fetched from the handle on first "
                               "access, so read them before close() / before leaving the `with` block")
        out = np.empty(shape, dtype=dtype)
        _lib.check(getattr(self._lib, fn)(self._handle, ctypes.c_void_p(out.ctypes.data)))
        return out

    def commit_log(self, instance, author):
        """``committed_history()`` of one node as a list of ``(proposer, index, time)``."""
        n = ctypes.c_size_t(0)
        _lib.check(self._lib.lbft_commit_log(self._handle, instance, author, None, 0, ctypes.byref(n)))
        buf = (_lib.LbftCommit * max(1, n.value))()
        _lib.check(self._lib.lbft_commit_log(self._handle, instance, author, buf, n.value, ctypes.byref(n)))
        return [(int(buf[i].proposer), int(buf[i].index), int(buf[i].time)) for i in range(n.value)]

    def commit_logs(self, cap=None):
        """``lbft_commit_logs``: every ``committed_history()`` of the batch with one device pass and one copy.  Returns
        ``(rows, lens)``: ``rows[instance, k]`` (fields ``proposer``, ``index``, ``time``) is row k of the instance's longest
        log and node n's log is ``rows[instance, :lens[instance, n]]``."""
        lens = np.empty((self.num_instances, self.num_nodes), dtype=np.uint32)
        if cap is None:
            cap = max(1, int(self._fetch("lbft_commit_counts", np.uint32, (self.num_instances, self.num_nodes)).max()))
        rows = np.empty((self.num_instances, int(cap)), dtype=COMMIT_DTYPE)
        _lib.check(self._lib.lbft_commit_logs(self._handle, ctypes.c_void_p(rows.ctypes.data), int(cap), ctypes.c_void_p(lens.ctypes.data)))
        return rows, lens

    def round_switches(self, instance):
        """``DataWriter::nodes_round_switch`` of one instance as ``[(node, round, time)]``, node-major
        (needs ``record_round_switches=True``)."""
        n = ctypes.c_size_t(0)
        _lib.check(self._lib.lbft_round_switches(self._handle, instance, None, 0, ctypes.byref(n)))
        buf = (_lib.LbftRoundSwitch * max(1, n.value))()
        _lib.check(self._lib.lbft_round_switches(self._handle, instance, buf, n.value, ctypes.byref(n)))
        return [(int(buf[i].node), int(buf[i].round), int(buf[i].time)) for i in range(n.value)]

    def write_data_files(self, path, instance=0):
        """``DataWriter::new`` + ``write_to_file`` (data_writer.rs:20-33, 61-96) for one instance:
        ``<path>/round_switches.txt`` and ``<path>/number_of_messages.txt``."""
        counters = self._fetch("lbft_counters", np.uint32, (self.num_instances, 12))[instance]
        write_data_files(path, self.num_nodes, self.round_switches(instance), int(counters[0]) + int(counters[1]) + int(counters[2]))


def format_round_switches_csv(num_nodes, switches):
    """Text of ``round_switches.txt`` (data_writer.rs:61-86) from ``[(node, round, time)]``.

    A header ``node 0,node 1,..`` then one row per round in ``0..max_round`` — EXCLUSIVE of the largest round any
    node reached, as the reference's ``for round_num in 0..max_round`` has it — holding, per node, the time at which
    that round was first seen, or nothing.  Text conventions are the ``csv`` crate's defaults (bft-lib/Cargo.toml:23
    ``csv = "1.1"``: ``,`` delimiter, ``\n`` terminator, quotes only when needed; a record that is a single empty field
    is written as ``""``).  FORMAT UNPINNED: neither the crate nor a Rust toolchain is available here, so the bytes
    are a restatement; the values are checked bit-exactly against the oracle, and the file is checked to read back
    through the steps of the reference's own consumer (visualization/round_switch/round_plotter.py:11-14, 52-53).
    """
    first = {}
    max_round = 0
    for node, rnd, time in switches:
        first.setdefault((node, rnd), time)  # `.find(..)`: the first entry of that round
        max_round = max(max_round, rnd)
    lines = [",".join("node %d" % n for n in range(num_nodes))]
    for rnd in range(max_round):
        fields = ["" if (n, rnd) not in first else str(first[(n, rnd)]) for n in range(num_nodes)]
        lines.append('""' if fields == [""] else ",".join(fields))
    return "\n".join(lines) + "\n"


def write_data_files(path, num_nodes, switches, message_count):
    if not os.path.exists(path):
        os.mkdir(path)  # fs::create_dir: not recursive (data_writer.rs:28-30)
    with open(os.path.join(path, "round_switches.txt"), "w", newline="") as f:
        f.write(format_round_switches_csv(num_nodes, switches))
    with open(os.path.join(path, "number_of_messages.txt"), "w", newline="") as f:
        f.write("%d\n" % message_count)  # wtr.serialize(Some(message_counter)) data_writer.rs:88-95


class Simulator:
    """Single-instance spelling of ``bft_lib::simulator::Simulator`` (simulator.rs:200-208, 380).

    ``context_factory`` is accepted for signature compatibility with the reference's callers
    (main.rs:23-34, simulated_run.rs:29-42); it may be ``None`` or a ``NodeConfig`` /
    ``(NodeConfig, commands_per_epoch)`` describing what the reference's closure would build.
    """

    def __init__(self, rng_seed, num_nodes, network_delay, context_factory=None, horizon=None, **kw):
        node_config, cpe = NodeConfig(), 30000
        # horizon: the largest clock any later loop_until will be given.  The reference needs no such thing (its heap is
        # unbounded); the device tables are sized for it.  Without it loop_until is one-shot, as before.
        self._horizon = None if horizon is None else int(horizon)
        self._ran = False
        if horizon is not None:
            kw["resumable"] = True
        if isinstance(context_factory, NodeConfig):
            node_config = context_factory
        elif isinstance(context_factory, tuple):
            node_config, cpe = context_factory
        elif context_factory is not None:
            raise TypeError("context_factory must be None, a NodeConfig or (NodeConfig, commands_per_epoch)")
        self._batch = BatchSimulator([rng_seed], num_nodes, network_delay, node_config, cpe, **kw)

    @staticmethod
    def new(rng_seed, num_nodes, network_delay, context_factory=None, horizon=None, **kw):
        return Simulator(rng_seed, num_nodes, network_delay, context_factory, horizon, **kw)

    def loop_until(self, max_clock, csv_path=None):
        if self._horizon is None:
            if self._ran:
                raise RuntimeError("loop_until was already run: pass horizon=<largest clock> to Simulator.new to call it again "
                                   "(the device tables are sized for a horizon, include/lbft.h lbft_run_until)")
            res = self._batch.loop_until(int(max_clock), csv_path)
        else:
            # simulator.rs:380 called repeatedly on one Simulator.  A DataWriter lives for ONE call (:381, :470-472), the
            # device keeps one table per run: csv_path is only supported on one-shot simulators.
            if csv_path is not None:
                raise ValueError("csv_path on a resumable Simulator is not supported")
            if not self._ran:
                self._batch.create(self._horizon)
            res = self._batch.run_until(int(max_clock))
        self._ran = True
        self.result = res
        return res.contexts(0)
