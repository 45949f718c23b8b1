"""The path bench.py times, compared with the oracle in the configuration it times.

The headline step is sym2_kernel (the symmetric-group fold), the fused truncation, the Instruction-record drain with
JR_STAGING_DEPTH batches in flight (a speculative DMA copy plus a tail fetch) and the host fold (jr_fsm_fold_mt).  The
digest-based parity suites never see the fold: JR_F_STREAM_DIGEST switches it off.  Here the engines are built like
bench.py's steady_engine (JR_F_CAPTURE_FSM only), and after every step the expanded Instruction stream must equal the
oracle's byte for byte, next to state digest, leader table, fault count and sampled replica state and block tables.

  A. case_bench_fold        the device-resident arm: jr_run + a drain per step, every group folded (and one mixed step)
  B. case_pipelined_drain   the end-to-end arm: jr_run_token_runs + jr_leader_table_async + jr_fsm_records_async with
                            three steps in flight, one step of arbitrary tokens that outgrows the speculative copy, the
                            host fold at several thread counts against a plain fold of the expanded stream; also with
                            the batches consumed on a second thread
  C. case_staging_contract  a returned batch stays intact until the JR_STAGING_DEPTH-1'th jr_fsm_records_async after
                            the wait, also when JR_STAGING_DEPTH batches were outstanding

Each case runs on the host build of the device code (tests/emu) at small sizes and on the GPU at the bench's sizes.
The constants come from bench.py, so these tests follow the bench if it changes."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

import bench
from josefine_b200 import abi
from tests import parity

S, DT = bench.TICKS_PER_STEP, bench.DT_MS
NB = 3                                                  # JR_STAGING_DEPTH: steps in flight on the async paths
INSTR = np.dtype([("group", "<u4"), ("node", "<u4"), ("kind", "u1"), ("client_kind", "u1"), ("reserved", "<u2"),
                  ("client_id", "<u4"), ("id", "<u8"), ("next", "<u8"), ("data", "<u8")])      # jr_fsm_instr
LEADER = np.dtype([("term", "<u8"), ("leader_id", "<u4"), ("commit", "<u4")])                  # jr_leader_entry
assert INSTR.itemsize == C.sizeof(abi.FsmInstr) and LEADER.itemsize == C.sizeof(abi.LeaderEntry)
FOLD_THREADS = (1, 2, 3, 8)


def _oracle(g, r, **kw):
    from oracle.restated import RestatedCluster
    return RestatedCluster.create(g, r, n_threads=min(16, os.cpu_count() or 1) if g >= 1024 else 1, **kw)


def _emu(g, r, **kw):
    from tests.emu.emu import EmuEngine
    return EmuEngine.create(g, r, **kw)


def _gpu(g, r, **kw):
    from josefine_b200 import RaftEngine
    return RaftEngine.create(g, r, **kw)


def _bind_async(lib):
    """argtypes of the asynchronous calls the Python wrapper does not use itself."""
    vp = C.c_void_p
    for name, args in (("jr_host_alloc", [C.c_size_t, C.POINTER(vp)]), ("jr_leader_table_async", [vp, vp]),
                       ("jr_leader_table_wait", [vp]), ("jr_engine_sync", [vp])):
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = args, C.c_int
    lib.jr_host_free.argtypes, lib.jr_host_free.restype = [vp], None


# ---------------------------------------------------------------------------------------------------------------------
# helpers

def bench_config(**over):
    """bench.py's steady_engine configuration (single rank)."""
    cfg = dict(seed=bench.SEED, chain_capacity=bench.CHAIN_WINDOW, flags=abi.F_CAPTURE_FSM, fsm_units=bench.FSM_UNITS,
               mailbox_units=64, heartbeat_ms=100)
    cfg.update(over)
    return cfg


def steady_pair(make, G, R, scattered=False, **over):
    """The engine and the oracle brought to the bench's steady state the way steady_engine does it: bootstrap, 16 ticks,
    truncate, the start-up stream discarded, fused truncation on."""
    cfg = bench_config(**over)
    eng, ora = make(G, R, **cfg), _oracle(G, R, **cfg)
    inj = bench.bootstrap_inject(G, R, scattered=scattered)
    for api in (eng, ora):
        api.step(0, flags=0, inject=inj)
        api.run(DT, DT, 16, 1)
        api.truncate(bench.TRUNC_MARGIN)
        api.discard_fsm(strict=False)
        api.set_auto_truncate(bench.TRUNC_MARGIN)
    return eng, ora


def fsm_cap(G, R, cfg):
    """Records one batch may hold (jr_config.fsm_host_records and its default, include/josefine_raft_abi.h)."""
    reps = G * R
    want = cfg.get("fsm_host_records") or max(3 * reps + 1024, min(reps * cfg["fsm_units"], 1 << 16))
    return min(want, 0x7fffffff)


def speculative_copy(last_records, cap):
    """Records jr_fsm_records_async copies before the batch size is known: the previous batch's size plus a margin."""
    return min(cap, max(last_records + last_records // 8 + 1024, 16384))


def wait_batch(lib, h):
    ptr, batch = C.POINTER(abi.FsmRecord)(), abi.FsmBatch()
    st = lib.jr_fsm_records_wait(h, C.byref(ptr), C.byref(batch))
    assert st == abi.OK, (st, batch.n_dropped)
    return ptr, batch


def record_words(ptr, n):
    """A copy of n jr_fsm_record (eight 32-bit words each) from the engine's buffer."""
    if n == 0:
        return np.zeros((0, 8), dtype=np.uint32)
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint32)), shape=(n * 8,)).reshape(n, 8).copy()


def expand(lib, words, G, R):
    """jr_fsm_expand of a record array -> jr_fsm_instr array."""
    n = len(words)
    recs = words.ctypes.data_as(C.POINTER(abi.FsmRecord))
    need = C.c_size_t(0)
    st = lib.jr_fsm_expand(recs, C.c_size_t(n), G, R, None, C.c_size_t(0), C.byref(need))
    assert st in (abi.OK, abi.E_CAPACITY), st
    out = np.zeros(need.value, dtype=INSTR)
    if need.value:
        st = lib.jr_fsm_expand(recs, C.c_size_t(n), G, R, out.ctypes.data_as(C.POINTER(abi.FsmInstr)), need, C.byref(need))
        assert st == abi.OK, st
    return out[:need.value]


def oracle_drain(ora, G, R, ticks):
    cap = G * (R + 1) * ticks + 8 * G * R + 1024
    out = np.zeros(cap, dtype=INSTR)
    n = C.c_size_t(0)
    st = ora._lib.jro_drain_fsm(ora._h, out.ctypes.data_as(C.POINTER(abi.FsmInstr)), C.c_size_t(cap), C.byref(n))
    assert st == abi.OK, st
    return out[:n.value]


def assert_same_stream(got, want, where):
    if len(got) == len(want) and np.array_equal(got.view(np.uint8), want.view(np.uint8)):
        return
    n = min(len(got), len(want))
    bad = np.nonzero(got[:n] != want[:n])[0]
    i = int(bad[0]) if len(bad) else n
    pytest.fail(f"{where}: the engine's expanded stream ({len(got)} Instructions) differs from the oracle's ({len(want)}); "
                f"first difference at #{i}: engine {got[i] if i < len(got) else None}, oracle {want[i] if i < len(want) else None}")


def check_batch(words, batch, n_instructions, G, R):
    """The batch header describes the records, and the records are sorted by (node, group)."""
    n = len(words)
    assert (batch.n_records, batch.n_dropped, batch.n_instructions) == (n, 0, n_instructions)
    group, node = words[:, 0], ((words[:, 1] >> 2) & 7) + 1
    assert n == 0 or (group.max() < G and node.max() <= R)
    key = (node.astype(np.uint64) << np.uint64(32)) | group.astype(np.uint64)
    assert np.all(key[1:] >= key[:-1]), "records are not sorted by (node, group)"
    off = [batch.node_offset[r] for r in range(R + 1)]
    assert off == sorted(off) and off[0] == 0 and off[R] == n
    assert list(np.searchsorted(node, np.arange(1, R + 1), side="right")) == off[1:], "node_offset does not match the records"


def compare_sampled(eng, ora, groups, where):
    """Exact replica state and the block-table rows above the floor, on a sample of groups."""
    R = eng.n_replicas
    parity.compare_states(eng, ora, groups=groups, where=where)
    reqs = [(g, n, int(eng.query(g, n).chain_floor), 24) for g in groups for n in range(1, R + 1)]
    assert eng.chain_read_many(reqs) == ora.chain_read_many(reqs), f"{where} block tables differ"


def sample_groups(G, extra=()):
    if G <= 256:
        return list(range(G))
    return sorted(set(range(0, G, 4099)) | {1, 63, 64, 4095, 4096, G // 2, G - 1} | set(extra))


# ---------------------------------------------------------------------------------------------------------------------
# A. the device-resident arm: sym2_kernel at the bench's configuration

def case_bench_fold(make, G, R, steps=3, scattered=False, heartbeat_ms=100, group_offset=0, mixed_after=None):
    """bench.py's device-resident step (jr_run of 64 ticks with one synthetic proposal per tick, fused truncation, one
    drain per step) on an engine that folds, against the oracle, step after step.  With `mixed_after`, one follower is
    silenced in ~1% of the groups before that step: the launch then has CTAs with folded and unfolded groups, and it
    starts with the stale hint that every group folded (so step_kernel is launched in one part).  Returns the fold
    counts and the silenced groups."""
    eng, ora = steady_pair(make, G, R, scattered=scattered, heartbeat_ms=heartbeat_ms, group_offset=group_offset)
    lib, h = eng._lib, eng._h
    now, folds, silenced = DT * 17, [], []
    for k in range(steps):
        if k == mixed_after:
            silenced = list(range(0, G, 100))
            for g in silenced:
                leader = g % R + 1 if scattered else 1
                for api in (eng, ora):
                    api.set_alive(g, leader % R + 1, False)
        for api in (eng, ora):
            api.run(now, DT, S, 1)
        now += DT * S
        folds.append(eng.fold_count())
        where = f"[{G}x{R} step {k}, {folds[-1]} groups folded]"
        assert lib.jr_fsm_records_async(h) == abi.OK
        ptr, batch = wait_batch(lib, h)
        words = record_words(ptr, batch.n_records)
        got, want = expand(lib, words, G, R), oracle_drain(ora, G, R, S)
        assert_same_stream(got, want, where)
        assert len(want) >= G * (R + 1) * (S - 2), (where, len(want))       # every group commits a block per tick
        check_batch(words, batch, len(want), G, R)
        assert eng.state_digest() == ora.state_digest(), f"{where} state digest differs"
        assert eng.leader_table() == ora.leader_table(), f"{where} leader table differs"
        assert eng.fault_count() == ora.fault_count() == 0, where
        compare_sampled(eng, ora, sample_groups(G, silenced[:4]), where)
    return folds, silenced


@pytest.mark.parametrize("R", [5, 3])
def test_bench_fold_on_device_code(R):
    """G = 130: two full CTAs of sym2_kernel and a partial one.  R = 5 ends with a mixed step."""
    mixed = 2 if R == 5 else None
    folds, silenced = case_bench_fold(_emu, 130, R, steps=3, mixed_after=mixed)
    assert folds[:2] == [130, 130], folds
    if mixed is None:
        assert folds[2] == 130, folds
    else:
        assert silenced == [0, 100] and 0 < folds[2] <= 130 - len(silenced), folds


def test_bench_fold_heartbeat_99_on_device_code():
    folds, _ = case_bench_fold(_emu, 130, 5, steps=3, heartbeat_ms=99)
    assert folds == [130] * 3, folds


@pytest.mark.gpu
def test_bench_fold_65536x5_on_gpu():
    """The headline: 65,536 x 5, leaders on node 1, 1,024 CTAs of sym2_kernel in one wave; then a mixed step."""
    G = bench.GROUPS_PER_GPU
    folds, silenced = case_bench_fold(_gpu, G, bench.REPLICAS, steps=3, mixed_after=2)
    assert folds[:2] == [G, G], folds
    assert 0 < folds[2] <= G - len(silenced), folds


@pytest.mark.gpu
def test_bench_fold_65536x5_scattered_leaders_on_gpu():
    G = bench.GROUPS_PER_GPU
    folds, _ = case_bench_fold(_gpu, G, bench.REPLICAS, steps=3, scattered=True)
    assert folds == [G] * 3, folds


@pytest.mark.gpu
def test_bench_fold_65536x5_heartbeat_99_on_gpu():
    G = bench.GROUPS_PER_GPU
    folds, _ = case_bench_fold(_gpu, G, bench.REPLICAS, steps=3, heartbeat_ms=99)
    assert folds == [G] * 3, folds


@pytest.mark.gpu
def test_bench_fold_131072x5_group_offset_on_gpu():
    """A 131,072-group shard (BASELINE config #4, second rank): sym2_kernel runs two waves of CTAs."""
    G = 2 * bench.GROUPS_PER_GPU
    folds, _ = case_bench_fold(_gpu, G, bench.REPLICAS, steps=3, group_offset=G)
    assert folds == [G] * 3, folds


@pytest.mark.gpu
def test_bench_fold_65536x7_on_gpu():
    G = bench.GROUPS_PER_GPU
    folds, _ = case_bench_fold(_gpu, G, 7, steps=3)
    assert folds == [G] * 3, folds


# ---------------------------------------------------------------------------------------------------------------------
# B. the end-to-end arm: three steps in flight through the C ABI

class HostFold:
    """jr_fsm_fold_mt at several thread counts, and a plain fold of the expanded Instructions to compare them with:
    per (node, group) the highest block id applied; Apply, Notify and record counts."""

    def __init__(self, lib, G, R):
        self.lib, self.G, self.R = lib, G, R
        self.applied = {t: np.zeros(G * R, dtype=np.uint32) for t in FOLD_THREADS}
        self.totals = {t: np.zeros(3, dtype=np.uint64) for t in FOLD_THREADS}
        self.ref_applied, self.ref_totals = np.zeros(G * R, dtype=np.uint32), np.zeros(3, dtype=np.uint64)

    def fold(self, ptr, n):
        """Folds the batch where jr_fsm_records_wait left it."""
        for t in FOLD_THREADS:
            st = self.lib.jr_fsm_fold_mt(C.cast(ptr, C.c_void_p), C.c_size_t(n), self.G, self.R,
                                         self.applied[t].ctypes.data, self.totals[t].ctypes.data, t)
            assert st == abi.OK, (t, st)

    def reference(self, instr, n_records):
        apply = instr[instr["kind"] == abi.FSM_APPLY]
        np.maximum.at(self.ref_applied, (apply["node"].astype(np.int64) - 1) * self.G + apply["group"], apply["id"].astype(np.uint32))
        self.ref_totals += np.array([len(apply), np.count_nonzero(instr["kind"] == abi.FSM_NOTIFY), n_records], dtype=np.uint64)

    def check(self, where):
        for t in FOLD_THREADS:
            assert list(self.totals[t]) == list(self.ref_totals), f"{where} jr_fsm_fold_mt({t} threads) totals"
            bad = np.nonzero(self.applied[t] != self.ref_applied)[0]
            assert len(bad) == 0, (f"{where} jr_fsm_fold_mt({t} threads): {len(bad)} watermarks differ, first (node "
                                   f"{bad[0] // self.G + 1}, group {bad[0] % self.G}): {self.applied[t][bad[0]]} vs {self.ref_applied[bad[0]]}")


def case_pipelined_drain(make, G, R, steps=8, arbitrary_at=4, arbitrary_ticks=S, two_threads=False, **over):
    """Per step, as bench.py's end-to-end arm submits it: jr_run_token_runs (pinned jr_token_run[3][G]), then
    jr_leader_table_async (pinned jr_leader_entry[3][G]), then jr_fsm_records_async; three steps in flight, the oldest
    consumed.  Step `arbitrary_at` is a jr_run_tokens of arbitrary tokens instead: one record per Instruction, a batch
    larger than the speculative copy, so jr_fsm_records_wait fetches the tail.  The oracle runs the same steps one at a
    time; every batch must expand to its drain, every leader table equal its leader table, and the host fold agree with a
    plain fold of the expanded stream.  With `two_threads`, a second thread consumes and follows the header's rule to
    the letter: the submitting thread may go on as soon as jr_fsm_records_wait has returned, and the consumer reads the
    batch until it waits for the next one (before the JR_STAGING_DEPTH-1'th jr_fsm_records_async after its wait)."""
    cfg = bench_config(**over)
    eng, ora = steady_pair(make, G, R, **over)
    lib, h = eng._lib, eng._h
    _bind_async(lib)
    cap = fsm_cap(G, R, cfg)
    for api in (eng, ora):
        api.leader_table()                                   # first announce: where the tokens go
    bufs = []
    for _ in range(2):
        p = C.c_void_p()
        assert lib.jr_host_alloc(C.c_size_t(NB * G * 16), C.byref(p)) == abi.OK
        bufs.append(p.value)
    runs = np.ctypeslib.as_array((C.c_uint64 * (NB * G * 2)).from_address(bufs[0])).reshape(NB, G, 2)
    tables = np.ctypeslib.as_array((C.c_uint8 * (NB * G * 16)).from_address(bufs[1])).view(LEADER).reshape(NB, G)
    rng = np.random.default_rng(7)

    def plan(k):
        """Step k: (ticks, run-length bases or None, arbitrary tokens or None, now)."""
        ticks = arbitrary_ticks if k == arbitrary_at else S
        now = DT * 17 + DT * (S * k + (arbitrary_ticks - S if k > arbitrary_at else 0))
        if k == arbitrary_at:
            return ticks, None, rng.integers(1, 1 << 63, size=(ticks, G), dtype=np.uint64), now
        return ticks, (np.uint64(k * S + 1) << np.uint64(32)) + np.arange(G, dtype=np.uint64), None, now

    plans = [plan(k) for k in range(steps)]
    n_records, guesses = [], {}
    last_taken = [None]           # n_records of the batch jr_fsm_records_wait returned last (single-thread order)
    fold = HostFold(lib, G, R)
    fail = []

    def submit(k):
        ticks, bases, tokens, now = plans[k]
        if bases is not None:
            runs[k % NB, :, 0], runs[k % NB, :, 1] = bases, 1 << 32     # buffer k % NB: its step k - 3 has been consumed
            st = lib.jr_run_token_runs(h, C.c_uint64(now), C.c_uint32(DT), C.c_uint32(ticks),
                                       C.cast(bufs[0] + (k % NB) * G * 16, C.POINTER(abi.TokenRun)))
        else:                                                # pageable: the call blocks for the copy
            st = lib.jr_run_tokens(h, C.c_uint64(now), C.c_uint32(DT), C.c_uint32(ticks), tokens.ctypes.data_as(C.POINTER(C.c_uint64)))
        assert st == abi.OK, st
        assert lib.jr_leader_table_async(h, C.c_void_p(bufs[1] + (k % NB) * G * 16)) == abi.OK
        if last_taken[0] is not None:
            guesses[k] = speculative_copy(last_taken[0], cap)
        assert lib.jr_fsm_records_async(h) == abi.OK

    def take(k):
        """Waits for step k's leader table and records; returns (table, records pointer, batch)."""
        assert lib.jr_leader_table_wait(h) == abi.OK
        table = tables[k % NB].copy()
        ptr, batch = wait_batch(lib, h)
        n_records.append(batch.n_records)
        last_taken[0] = batch.n_records
        return table, ptr, batch

    def check(k, table, ptr, batch):
        """Everything that reads the engine's buffer; then the oracle's step k and the comparison."""
        where = f"[{G}x{R} step {k}{' (arbitrary tokens)' if k == arbitrary_at else ''}]"
        fold.fold(ptr, batch.n_records)
        words = record_words(ptr, batch.n_records)
        got = expand(lib, words, G, R)
        ticks, bases, tokens, now = plans[k]
        if bases is not None:
            ora.run_token_runs(now, DT, ticks, [(int(b), 1 << 32) for b in bases])
        else:
            assert ora._lib.jro_run_tokens(ora._h, C.c_uint64(now), C.c_uint32(DT), C.c_uint32(ticks),
                                           tokens.ctypes.data_as(C.POINTER(C.c_uint64))) == abi.OK
        want_table = ora.leader_table()
        want = oracle_drain(ora, G, R, ticks)
        assert_same_stream(got, want, where)
        check_batch(words, batch, len(want), G, R)
        assert [(int(e["term"]), int(e["leader_id"]), int(e["commit"])) for e in table] == want_table, f"{where} leader table"
        fold.reference(want, batch.n_records)
        fold.check(where)

    try:
        if not two_threads:
            for k in range(NB - 1):
                submit(k)
            for k in range(steps):
                if k + NB - 1 < steps:
                    submit(k + NB - 1)
                check(k, *take(k))
        else:
            free, ready, stop = threading.Semaphore(NB), threading.Semaphore(0), []

            def consumer():
                try:
                    for k in range(steps):
                        ready.acquire()
                        if stop:
                            return
                        got = take(k)
                        free.release()               # the batch stays valid until the second jr_fsm_records_async after this
                        check(k, *got)
                except BaseException as ex:          # noqa: BLE001 -- handed to the submitting thread
                    fail.append(ex)
                    for _ in range(steps + NB):
                        free.release()

            th = threading.Thread(target=consumer, name="fsm-driver")
            th.start()
            try:
                for k in range(steps):
                    free.acquire()
                    if fail:
                        break
                    submit(k)
                    ready.release()
            except BaseException:
                stop.append(True)
                ready.release()
                raise
            finally:
                th.join()
            if fail:
                raise fail[0]
    finally:
        lib.jr_engine_sync(h)
        for p in bufs:
            lib.jr_host_free(C.c_void_p(p))
    n_arb = n_records[arbitrary_at]
    assert n_arb <= cap
    if two_threads:          # the wait that ran last before the submit is one of the three before it
        guess = max(speculative_copy(n, cap) for n in n_records[arbitrary_at - NB:arbitrary_at])
    else:
        guess = guesses[arbitrary_at]
        assert guess == speculative_copy(n_records[arbitrary_at - NB], cap)
    assert n_arb > guess, f"the arbitrary-token batch ({n_arb} records) fits the speculative copy ({guess}): no tail fetch"
    assert eng.state_digest() == ora.state_digest() and eng.fault_count() == ora.fault_count() == 0
    compare_sampled(eng, ora, sample_groups(G), f"[{G}x{R} end]")
    return n_records


def test_pipelined_drain_on_device_code():
    """G = 256, R = 5: 64 ticks of arbitrary tokens make ~95 records per group (the leader's Apply and Notify runs are one
    Instruction long; the followers share theirs through the fold), ~24,000 in all: more than the smallest speculative
    copy (16,384 records)."""
    n = case_pipelined_drain(_emu, 256, 5, fsm_units=256)
    assert n[4] > 16384 and max(n[:4] + n[5:]) < 4096, n


def test_pipelined_drain_two_threads_on_device_code():
    n = case_pipelined_drain(_emu, 256, 5, fsm_units=256, two_threads=True)
    assert n[4] > 16384, n


@pytest.mark.gpu
def test_pipelined_drain_65536x5_on_gpu():
    """At the bench's size.  12 ticks of arbitrary tokens (some 40 records per group, far past the speculative copy) fit
    a FIFO of 64 records per replica and a batch of 24 records per replica, also where a group leaves the fold."""
    G, R = bench.GROUPS_PER_GPU, bench.REPLICAS
    n = case_pipelined_drain(_gpu, G, R, arbitrary_ticks=12, fsm_units=64, fsm_host_records=G * R * 24)
    assert n[4] > 2 * max(n[:4]), n


@pytest.mark.gpu
def test_pipelined_drain_two_threads_65536x5_on_gpu():
    G, R = bench.GROUPS_PER_GPU, bench.REPLICAS
    case_pipelined_drain(_gpu, G, R, steps=6, arbitrary_at=3, arbitrary_ticks=12, fsm_units=64,
                         fsm_host_records=G * R * 24, two_threads=True)


# ---------------------------------------------------------------------------------------------------------------------
# C. the staging contract

def case_staging_contract(make, G, R):
    """JR_STAGING_DEPTH batches outstanding, then jr_fsm_records_wait: the buffer it returns must not change through the
    next jr_fsm_records_async (it is the caller's until the one after).  Every batch also equals the oracle's drain."""
    eng, ora = steady_pair(make, G, R)
    lib, h = eng._lib, eng._h
    _bind_async(lib)
    want = []
    now = DT * 17
    for _ in range(NB):
        for api in (eng, ora):
            api.run(now, DT, S, 1)
        now += DT * S
        want.append(oracle_drain(ora, G, R, S))
        assert lib.jr_fsm_records_async(h) == abi.OK
    ptr, batch = wait_batch(lib, h)
    snap = record_words(ptr, batch.n_records)
    for api in (eng, ora):
        api.run(now, DT, S, 1)
    want.append(oracle_drain(ora, G, R, S))
    assert lib.jr_fsm_records_async(h) == abi.OK
    assert lib.jr_engine_sync(h) == abi.OK
    after = record_words(ptr, batch.n_records)
    changed = int(np.count_nonzero((after != snap).any(axis=1)))
    assert changed == 0, f"{changed} of {batch.n_records} records of the returned batch changed under the next jr_fsm_records_async"
    assert_same_stream(expand(lib, snap, G, R), want[0], "batch 0")
    for k in range(1, NB + 1):
        ptr, batch = wait_batch(lib, h)
        words = record_words(ptr, batch.n_records)
        got = expand(lib, words, G, R)
        assert_same_stream(got, want[k], f"batch {k}")
        check_batch(words, batch, len(want[k]), G, R)
    assert eng.state_digest() == ora.state_digest()


def test_staging_contract_on_device_code():
    case_staging_contract(_emu, 64, 5)


@pytest.mark.gpu
def test_staging_contract_65536x5_on_gpu():
    case_staging_contract(_gpu, bench.GROUPS_PER_GPU, bench.REPLICAS)
