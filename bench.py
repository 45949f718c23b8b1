#!/usr/bin/env python
"""bench.py -- Raft-group ticks/sec of the batched Chained-Raft step path.

Metric (BASELINE.json): Raft-group ticks/sec @ 64Ki groups x 5 replicas.
One group-tick = all R replicas of one group each drain the peer mail of the
previous step, take the step's client proposal (leader) and apply one
Command::Tick (SURVEY.md section 8d; the reference defines no such unit -- its
Tick is a 100 ms wall-clock interval, src/raft/server.rs:25).

Headline workload (config.workload): BASELINE config #3 -- 65,536 groups x 5 replicas
per GPU, leaders pre-elected on node 1 by a synthetic vote trace, then steady state:
one client proposal per group per tick, AppendEntries / AppendResponse / Heartbeat /
HeartbeatResponse traffic between the co-resident replicas.  heartbeat_ms = tick = 100 ms
and the reference compares with a strict `>` (leader.rs:78-84), so the leader heartbeats
every SECOND tick; `variants.heartbeat_every_tick` (heartbeat_ms = 99) is the other reading.

A bench "step" = TICKS_PER_STEP consecutive group-ticks of every group: one fused call
(jr_run / jr_run_token_runs) that ends with jr_truncate (jr_set_auto_truncate; deviation D7:
the block-table window moves up, so an engine runs indefinitely -- no reset anywhere in this
file), and the drain of the step's Instruction stream (jr_fsm_records_async: count + scan +
pack on the engine stream, DMA to pinned host memory on the copy stream).  L2 is flushed
between timed steps (the working set is smaller than the 126 MB L2).  Device time is taken
with CUDA events on the engine's stream, per step, flush excluded; max over ranks.

Arms:
  (default)          the CUDA engine.  `value` = device-resident throughput (proposals
                     generated in the kernel, Instruction stream drained every step);
                     `e2e` = the same workload through the C ABI with HOST buffers, every
                     step: the step's proposals H2D from pinned memory in run-length form
                     (jr_run_token_runs: {base, stride} per group), the per-group leader
                     table D2H, the step's Instruction records D2H and folded on the host;
                     three steps in flight (JR_STAGING_DEPTH).
                     `e2e_dense_input` = the same with one 8-byte token per group-tick
                     (jr_run_tokens, round 1's input); `e2e_no_output` = round 1's leg:
                     dense input, engine created without the Instruction stream.
                     `other_configs` = BASELINE configs #2, #4 (per-GPU shard) and #5, each
                     timed at its size; `parity` = state/stream digests against the C++
                     restatement on the same inputs, per config, in this run.
  --impl reference   the CPU comparator: the C++ RESTATEMENT of josefine's src/raft
                     (oracle/; josefine itself is Rust and cannot be built here) on the
                     host cores, the SAME config #3 workload at full size.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from josefine_b200 import abi, Command  # noqa: E402

METRIC = "Raft-group ticks/sec @ 64Ki groups x 5 replicas"   # BASELINE.json `metric`
UNIT = "group-ticks/s"
GROUPS_PER_GPU = 65536
REPLICAS = 5
TICKS_PER_STEP = 64
DT_MS = 100
SEED = 1
L2_FLUSH_BYTES = 256 << 20
CHAIN_WINDOW = 512          # block ids a replica's table may span above the floor (truncated every step)
TRUNC_MARGIN = 8
FSM_UNITS = 16              # record slots per replica between two drains (steady state uses <= 4)
FOLD_THREADS = int(os.environ.get("JR_FOLD_THREADS", "0"))   # host threads folding a batch of Instruction records (jr_fsm_fold_mt, groups partitioned
#                                                               over threads); 0 = what this rank's share of the usable host cores allows, at most 8


def workload_name(G, R):
    return (f"BASELINE config #3: {G} groups x {R} replicas per GPU, pre-elected leaders, steady-state "
            f"AppendEntries, 1 proposal/group/tick, {TICKS_PER_STEP} ticks per step")


_boot_cache = {}


def bootstrap_inject(G, R, node=1, scattered=False):
    """Synthetic vote trace: Timeout on `node` (or on node g % R + 1 with `scattered`), plus
    quorum-1 granted VoteResponses."""
    key = (G, R, node, scattered)
    if key not in _boot_cache:
        _boot_cache.clear()          # (one list at a time: ~200k ctypes structs each)
        _boot_cache[key] = _bootstrap_inject(G, R, node, scattered)
    return _boot_cache[key]


def _bootstrap_inject(G, R, node, scattered):
    q = 0 if R == 1 else R // 2 + 1
    inj = []
    for g in range(G):
        n = (g % R) + 1 if scattered else node
        inj.append(Command.timeout(g, n))
        for v in [v for v in range(1, R + 1) if v != n][:max(q - 1, 0)]:
            inj.append(Command.vote_response(g, n, 1, v, True))
    return inj


# ---------------------------------------------------------------------------------------------
# algorithmic bytes (DESIGN.md section 6)

def algorithmic_bytes_per_group_tick(make, R, ticks=64, heartbeat_ms=100):
    """Bytes one steady-state group-tick must move, from the message mix of a small captured run.
    Returns (reference_widths, layout):
      reference_widths  SURVEY.md 8(d): per replica state 40 B read + 40 B written; each message's decision fields
                        in the reference's own widths, written once and read once per addressee
                        (AppendEntries 16 + 16/block, AppendResponse 24, Heartbeat 20, HeartbeatResponse 12,
                        VoteRequest 28, VoteResponse 16, ClientRequest/Response 24); leader progress heads R x 8 B
                        read + written; block table 16 B per block appended / extended
      layout            the same count with THIS engine's widths (16 B mailbox units, 52/116 B state planes, 12 B table
                        rows, 32 B Instruction records) -- wider than the reference's, so it may not raise the claim
    """
    G = 32
    eng = make(G, R, seed=SEED, flags=abi.F_CAPTURE_MESSAGES | abi.F_CAPTURE_FSM, chain_capacity=ticks * 2 + 64,
               fsm_units=64, heartbeat_ms=heartbeat_ms)
    eng.step(0, flags=0, inject=bootstrap_inject(G, R))
    for k in range(16):  # reach the steady regime
        eng.step((k + 1) * DT_MS, n_synth=1)
    ref_w = {abi.CMD_APPEND_ENTRIES: 16, abi.CMD_APPEND_RESPONSE: 24, abi.CMD_HEARTBEAT: 20, abi.CMD_HEARTBEAT_RESPONSE: 12,
             abi.CMD_VOTE_REQUEST: 28, abi.CMD_VOTE_RESPONSE: 16, abi.CMD_CLIENT_REQUEST: 24, abi.CMD_CLIENT_RESPONSE: 24}
    tot_ref = tot_lay = 0
    for k in range(16, 16 + ticks):
        res = eng.step((k + 1) * DT_MS, n_synth=1)
        ref = G * R * 40 * 2 + G * R * 8 * 2                  # state R+W, progress heads R+W (one leader per group)
        lay = G * ((R - 1) * 52 + 116) * 2                    # state planes read + written
        lay += G * R * 4 * 2 + G * R * (R - 1) * 4            # mailbox counts: reset/written, read by each peer
        seen_vreq, seen_runs = set(), set()
        for m in res.messages:
            readers = (R - 1) if m.to_kind == abi.ADDR_PEERS else 1
            ref += (ref_w.get(m.kind, 8) + 16 * m.n_blocks) * (1 + readers)
            if m.kind == abi.CMD_APPEND_ENTRIES:
                ref += 16 * m.n_blocks                        # the follower's table rows
            if m.kind == abi.CMD_VOTE_REQUEST:                # N-1 copies share one unit
                key = (m.group, m.from_id)
                if key in seen_vreq:
                    continue
                seen_vreq.add(key)
            lay += 16 * (1 + readers)                         # header unit: written once, read per addressee
            if m.kind == abi.CMD_APPEND_ENTRIES and m.n_blocks:
                run = (m.group, m.from_id, tuple(m.blocks[i].id for i in range(m.n_blocks)))
                if run not in seen_runs:                      # identical block runs of one sender are emitted once
                    seen_runs.add(run)
                    lay += m.n_blocks * (12 + 16)             # leader reads the table entries, writes the block units
                lay += m.n_blocks * (16 + 4 + 12)             # each follower reads the units, probes has(next), writes its table
        for f in res.fsm:
            if f.kind == abi.FSM_NOTIFY:
                ref += 16                                     # the leader's append: one table row
            lay += 12                                         # Notify: block written by append; Apply: block read
        tot_ref += ref
        tot_lay += lay
    return tot_ref / (G * ticks), tot_lay / (G * ticks)


class ClockSampler:
    """nvidia-smi clocks and throttle reasons (profiling recipe's clocks line).  Started before
    the warm-up so nvidia-smi's start-up latency is absorbed; `window()` keeps the samples
    that arrived inside the timed region."""

    def __init__(self, index):
        self.index = index
        self.rows = []      # (arrival time, fields)
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def window(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0}
        time.sleep(0.1)
        self.proc.terminate()
        good = [(t, r) for t, r in self.rows if len(r) >= 6 and r[0].isdigit()]
        inside = [r for t, r in good if t0 <= t <= t1 + 0.03]
        where = "timed region"
        if not inside and good:   # region shorter than the sampling period: nearest samples under the same load
            good.sort(key=lambda tr: min(abs(tr[0] - t0), abs(tr[0] - t1)))
            inside = [r for _, r in good[:5]]
            where = "nearest to the timed region (region shorter than the 20 ms sampling period)"
        sm = [int(r[0]) for r in inside]
        mx = [int(r[1]) for r in inside if r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in inside for i in range(4) if r[2 + i].startswith("Active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "sampled": where}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, torch copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# host placement (VERDICT r1 weak #7 / next #9)

def bind_to_gpu_numa_node(index):
    """Run this process (and first-touch its pinned buffers) on the NUMA node the GPU hangs off."""
    info = {"gpu": index, "node": None, "cpus": None}
    try:
        bus = subprocess.check_output(["nvidia-smi", f"--id={index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                      text=True, stderr=subprocess.DEVNULL).strip().lower()
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info.update(node=node, cpus=len(cpus))
    except (OSError, ValueError, subprocess.CalledProcessError):
        pass
    return info


def effective_cores():
    """Host threads this process may really use: affinity mask and cgroup CPU quota, not just cpu_count()."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


# ---------------------------------------------------------------------------------------------
# CPU comparator: the C++ restatement (oracle/), NOT josefine

def cpu_cluster(G, R, threads, chain_window=CHAIN_WINDOW, heartbeat_ms=100, seed=SEED, flags=0):
    from oracle.restated import RestatedCluster
    c = RestatedCluster.create(G, R, n_threads=threads, seed=seed, chain_capacity=chain_window, heartbeat_ms=heartbeat_ms,
                               flags=flags)
    c.step(0, flags=0, inject=bootstrap_inject(G, R))
    c.run(DT_MS, DT_MS, 16, 1)
    c.truncate(TRUNC_MARGIN)
    return c


def best_cpu_threads(R, cores):
    """The restatement allocates heavily; more threads than the allocator / cgroup can feed makes it SLOWER.
    Probe a few counts on a small sample, once per host (cached under /tmp), and keep the fastest."""
    cache = f"/tmp/josefine_b200_cpu_threads_{cores}_{R}.json"
    try:
        return int(json.load(open(cache))["threads"])
    except (OSError, ValueError, KeyError):
        pass
    best, best_rate = 1, 0.0
    for th in sorted({1, 4, 8, 16, 32, 64, cores} & set(range(1, cores + 1))):
        g = max(512, 32 * th)
        c = cpu_cluster(g, R, th)
        t0 = time.perf_counter()
        c.run(DT_MS * 17, DT_MS, 32, 1)
        rate = g * 32 / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = th, rate
    try:
        json.dump({"threads": best}, open(cache, "w"))
    except OSError:
        pass
    return best


def cpu_steps(G, R, threads, n_steps):
    """Seconds per step of the config #3 workload on the restatement: the same calls the GPU arm makes."""
    c = cpu_cluster(G, R, threads)
    now = DT_MS * 17
    out = []
    for _ in range(n_steps):
        t0 = time.perf_counter()
        c.run(now, DT_MS, TICKS_PER_STEP, 1)
        c.truncate(TRUNC_MARGIN)
        out.append(time.perf_counter() - t0)
        now += DT_MS * TICKS_PER_STEP
    assert c.fault_count() == 0
    return out


def cpu_baseline_block(G, R, steps_best=5, steps_one=1):
    usable = effective_cores()
    threads = best_cpu_threads(R, usable)
    best = cpu_steps(G, R, threads, steps_best + 1)[1:]
    one = cpu_steps(G, R, 1, steps_one) if threads > 1 else best
    per_step = G * TICKS_PER_STEP
    sample = (f"{G} groups x {R} replicas x {TICKS_PER_STEP} ticks per step (the full config #3 step): median of {len(best)} steps at "
              f"{threads} threads, {len(one)} step at 1 thread; {usable} usable host threads")
    return {"value": per_step / statistics.median(best), "unit": UNIT, "cores": threads, "kind": "port",
            "value_1_thread": per_step / statistics.median(one), "sample": sample,
            "comparator": "C++ restatement of josefine src/raft (oracle/), NOT josefine itself (Rust, unbuildable here)"}


def run_reference(args):
    """--impl reference: the C++ restatement of src/raft on the host cores, config #3 at full size."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    G, R = args.groups, args.replicas
    usable = effective_cores()
    threads = best_cpu_threads(R, usable)
    times = cpu_steps(G, R, threads, args.warmup + args.steps)[args.warmup:]
    one = cpu_steps(G, R, 1, 1) if threads > 1 else times
    per_step = G * TICKS_PER_STEP
    value = per_step / statistics.median(times)
    sample = (f"{G} groups x {R} replicas x {TICKS_PER_STEP} ticks per step, median of {len(times)} steps at {threads} threads "
              f"(fastest of a cached probe over 1..{usable} usable host threads; groups partitioned statically)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": statistics.median(times) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(G, R), "groups_per_gpu": G, "replicas": R, "ticks_per_step": TICKS_PER_STEP,
                   "tick_ms": DT_MS, "seed": SEED,
                   "comparator": "C++ restatement of josefine src/raft (oracle/), NOT josefine itself (Rust, unbuildable here)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "value_1_thread": per_step / statistics.median(one)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path hands its caller, for comparing two builds output for output

DUMP_LIMIT_BYTES = 64 << 20


def fsm_record_words(ptr, n):
    """A batch of jr_fsm_record as an (n, 8) uint32 array: group, hdr, id0, addr, tok0 lo/hi, stride lo/hi.  Split into
    32-bit words, every field survives the float64 it is written as exactly."""
    import numpy as np
    if n == 0:
        return np.zeros((0, 8), dtype=np.uint32)
    words = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint32)), shape=(n, C.sizeof(abi.FsmRecord) // 4))
    return words.copy()


def write_outputs(path, outputs):
    """<path>/<name>.npy in float64 for every output (all values are integers below 2**53, so exact).  When the whole set
    is over DUMP_LIMIT_BYTES, the rows of the largest array are sampled: a seeded choice, kept in their original order,
    whose row numbers are written as <name>_rows.npy."""
    import numpy as np
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in outputs.items()}
    budget = DUMP_LIMIT_BYTES - 4096 * (len(arrays) + 1)          # (room for the .npy headers)
    if sum(a.nbytes for a in arrays.values()) > budget:
        name = max(arrays, key=lambda k: arrays[k].nbytes)
        a = arrays.pop(name)
        keep = (budget - sum(b.nbytes for b in arrays.values())) // (a.nbytes // len(a) + 8)   # a row + its row number
        rows = np.sort(np.random.default_rng(SEED).choice(len(a), size=keep, replace=False))
        arrays[name], arrays[name + "_rows"] = a[rows], rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


# ---------------------------------------------------------------------------------------------
# GPU arms

class Bench:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        torch.set_num_threads(1)      # no OpenMP team spinning next to the threads that feed and drain the engine
        self.torch, self.dist = torch, dist
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
        self.placement = bind_to_gpu_numa_node(self.local)     # before any pinned allocation (first touch)
        torch.cuda.set_device(self.local)
        if self.world > 1:
            # The 1 MB announce runs next to the step's drain kernels, never next to sym2_kernel (one_step below).
            # (NCCL's own channel count: capped at 2 the 2 x 1 MB all-gather took 134 us, at 1 channel 255 us)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        global FOLD_THREADS
        if FOLD_THREADS <= 0:     # the box's cgroup may allow far fewer cores than it shows, and the fold pool's workers spin between two
            #                       batches: stay clear of the quota (a throttled cgroup stalls every thread, the submitting one included)
            FOLD_THREADS = max(1, min(8, effective_cores() // self.world - 2))
        self.stream = torch.cuda.Stream()      # explicit non-default stream: handle 0 would mean "engine's own"
        torch.cuda.set_stream(self.stream)
        self.flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")

    def make(self, g, r, **kw):
        from josefine_b200 import RaftEngine
        kw.setdefault("device", self.local)
        e = RaftEngine.create(g, r, **kw)
        return e

    def steady_engine(self, G, R, flags, scattered=False, heartbeat_ms=100, seed=SEED, auto_truncate=True):
        e = self.make(G, R, seed=seed, group_offset=self.rank * G, chain_capacity=CHAIN_WINDOW, flags=flags,
                      fsm_units=FSM_UNITS, mailbox_units=64, heartbeat_ms=heartbeat_ms)
        e.set_stream(self.stream.cuda_stream)
        e.step(0, flags=0, inject=bootstrap_inject(G, R, scattered=scattered))
        e.run(DT_MS, DT_MS, 16, 1)
        e.truncate(TRUNC_MARGIN)
        if flags & abi.F_CAPTURE_FSM:
            e.discard_fsm(strict=False)      # the bootstrap's irregular start-up stream is not part of the workload
        if auto_truncate:
            e.set_auto_truncate(TRUNC_MARGIN)    # every fused run ends with jr_truncate(margin): same result as calling it, one pass less
        return e

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident: proposals generated in the kernel, Instruction stream drained every step
    def device_resident(self, G, R, steps, warmup, announce=True, sampler=None, keep_outputs=False, **eng_kw):
        torch, dist = self.torch, self.dist
        S = TICKS_PER_STEP
        capture = os.environ.get("JR_BENCH_CAPTURE", "1") != "0"      # diagnostic A/B only; the reported runs capture
        eng = self.steady_engine(G, R, abi.F_CAPTURE_FSM if capture else 0, **eng_kw)
        lib, h = eng._lib, eng._h
        now = [DT_MS * 17]
        world = self.world
        leaders = torch.empty(G * 16, dtype=torch.uint8, device="cuda")
        gathered = torch.empty(world * G * 16, dtype=torch.uint8, device="cuda") if world > 1 else None
        side = torch.cuda.Stream() if world > 1 else None
        announce_done = [None]
        totals = (C.c_uint64 * 3)()
        applied = (C.c_uint32 * (G * R))()
        outstanding = [0]
        outputs = {}

        def take(keep=False):
            # device-resident leg: the batch must have LANDED in pinned host memory, but it is not walked here (the
            # end-to-end leg folds every record; doing it here as well would make this leg measure the host)
            ptr, batch = C.POINTER(abi.FsmRecord)(), abi.FsmBatch()
            st = lib.jr_fsm_records_wait(h, C.byref(ptr), C.byref(batch))
            assert st == 0, (st, batch.n_dropped)
            totals[0] += batch.n_instructions
            totals[2] += batch.n_records
            outstanding[0] -= 1
            if keep:       # copied out of the engine's staging buffer, which a later jr_fsm_records_async reuses
                outputs["fsm_records"] = fsm_record_words(ptr, batch.n_records)
                outputs["fsm_batch"] = [batch.n_records, batch.n_dropped, batch.n_instructions, *batch.node_offset]

        def one_step():
            if world > 1 and announce and announce_done[0] is not None:
                # The previous announce must be over before the fused run starts: `leaders` is rewritten below, and sym2_kernel
                # needs 1,024 of the GPU's 1,036 CTA slots in ONE wave -- an NCCL kernel still holding two SMs would push CTAs
                # into a second wave and stretch the step by the collective's duration.
                self.stream.wait_event(announce_done[0])
            eng.run(now[0], DT_MS, S, 1)          # (ends with jr_truncate: jr_set_auto_truncate)
            now[0] += DT_MS * S
            if world > 1 and announce:
                # the one cross-shard exchange: leader announce, once per step (every 64 ticks).  The table is packed on the
                # engine stream right behind the run; the NCCL all-gather runs on a side stream, next to the drain below (and, in
                # this bench, the untimed L2 flush that follows); the last one of the timed region is waited for inside it.
                eng.leader_table_device(leaders.data_ptr())
                packed = torch.cuda.Event()
                packed.record(self.stream)
                with torch.cuda.stream(side):
                    side.wait_event(packed)
                    dist.all_gather_into_tensor(gathered, leaders)
                    ev = torch.cuda.Event()
                    ev.record(side)
                announce_done[0] = ev
            if capture:
                st = lib.jr_fsm_records_async(h)
                assert st == 0, st
                outstanding[0] += 1
                if outstanding[0] == 2:      # consume the PREVIOUS step's stream while this step runs
                    take()

        for _ in range(max(warmup, 3)):
            self.flush.fill_(1)
            one_step()
        while outstanding[0]:
            take()
        for k in range(3):
            totals[k] = 0
        self.barrier()
        t0 = time.time()
        evs = []
        for i in range(steps):
            self.flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(self.stream)
            one_step()
            if world > 1 and announce and i == steps - 1:
                self.stream.wait_event(announce_done[0])            # the last announce is not hidden by a next step: time it
            b.record(self.stream)
            evs.append((a, b))
        while outstanding[0]:
            take(keep=keep_outputs and capture and outstanding[0] == 1)      # the last batch is the last timed step's
        self.barrier()
        clocks = sampler.window(t0, time.time()) if sampler else None
        per = [a.elapsed_time(b) for a, b in evs]
        ms = self.max_over_ranks(sum(per))
        faults = eng.fault_count()
        table = eng.leader_table()
        commit_min = min(c for (_, _, c) in table)
        assert faults == 0, f"{faults} replicas faulted during the timed region"
        collective_us = None
        if world > 1 and announce:          # the collective alone, no kernel next to it
            cev = []
            with torch.cuda.stream(side):
                for _ in range(12):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(side)
                    dist.all_gather_into_tensor(gathered, leaders)
                    b.record(side)
                    cev.append((a, b))
            torch.cuda.synchronize()
            collective_us = statistics.median(a.elapsed_time(b) for a, b in cev[2:]) * 1e3
        res = {"ms_total": ms, "ms_per_step": ms / steps, "value": world * G * S * steps / (ms * 1e-3), "folded_groups_last_step": eng.fold_count(),
               "faulted_replicas": faults, "commit_min": commit_min, "instructions": int(totals[0] + totals[1]),
               "records": int(totals[2]), "collective_us": collective_us, "clocks": clocks,
               "ms_per_step_rank_median": statistics.median(per)}
        if keep_outputs:
            outputs["leader_table"] = table
            res["outputs"] = outputs
        del eng
        torch.cuda.empty_cache()
        return res

    # ---- end to end through the C ABI with host buffers
    def end_to_end(self, G, R, steps, warmup, with_output=True, dense_input=False):
        torch = self.torch
        S = TICKS_PER_STEP
        eng = self.steady_engine(G, R, abi.F_CAPTURE_FSM if with_output else 0)
        lib, h = eng._lib, eng._h
        NB = 3          # steps in flight (JR_STAGING_DEPTH): the copy-out and host fold of step k overlap steps k+1 and k+2
        prop = torch.zeros(NB, S, G, dtype=torch.int64).pin_memory()      # tokens[NB][S][G], one proposal per group-tick
        table = torch.zeros(NB, G, 2, dtype=torch.int64).pin_memory()     # jr_leader_entry[NB][G]
        prop[...] = ((torch.arange(NB * S, dtype=torch.int64).view(NB, S, 1) + 1) << 32) + torch.arange(G, dtype=torch.int64)
        # the same proposals in run-length form: jr_token_run[NB][G] = {base, stride}; tick k proposes base + k * stride
        runs = torch.zeros(NB, G, 2, dtype=torch.int64).pin_memory()
        runs[:, :, 1] = 1 << 32
        for b in range(NB):
            runs[b, :, 0] = ((b * S + 1) << 32) + torch.arange(G, dtype=torch.int64)
        runs_np = runs.numpy()        # same pinned memory; numpy's in-place add stays on this thread
        if not dense_input:
            del prop
        pstride, tstride, rstride = S * G * 8, G * 16, G * 16
        eng.leader_table()                                                 # first announce: where the tokens go
        now = [DT_MS * 17]
        totals = (C.c_uint64 * 3)()
        applied = (C.c_uint32 * (G * R))()
        rec_bytes = [0]
        checks = []

        def submit(i):
            k = seq[0]
            seq[0] += 1
            if dense_input:
                st = lib.jr_run_tokens(h, C.c_uint64(now[0]), C.c_uint32(DT_MS), C.c_uint32(S),
                                       C.cast(prop.data_ptr() + (i % NB) * pstride, C.POINTER(C.c_uint64)))   # H2D + route + fused kernel
            else:
                if k >= NB:   # (buffer k % NB was copied up when step k - NB started, and that step has been consumed)
                    runs_np[k % NB, :, 0] += (NB * S) << 32       # the host's next quantum of request numbers: tokens never repeat
                st = lib.jr_run_token_runs(h, C.c_uint64(now[0]), C.c_uint32(DT_MS), C.c_uint32(S),
                                           C.cast(runs.data_ptr() + (k % NB) * rstride, C.POINTER(abi.TokenRun)))   # 16 B per group H2D
            assert st == 0, st
            now[0] += DT_MS * S
            st = lib.jr_leader_table_async(h, C.cast(table.data_ptr() + (i % NB) * tstride, C.POINTER(abi.LeaderEntry)))   # result D2H
            assert st == 0, st
            if with_output:
                assert lib.jr_fsm_records_async(h) == 0                   # Instruction stream D2H

        trace = {"submit": 0.0, "table_wait": 0.0, "records_wait": 0.0, "fold": 0.0} if os.environ.get("JR_BENCH_TRACE") else None

        def consume(i):
            t0 = time.perf_counter()
            assert lib.jr_leader_table_wait(h) == 0
            checks.append(int(table[i % NB, 0, 1].item() >> 32))        # read the step's result: commit of group 0
            t1 = time.perf_counter()
            if with_output:
                ptr, batch = C.POINTER(abi.FsmRecord)(), abi.FsmBatch()
                st = lib.jr_fsm_records_wait(h, C.byref(ptr), C.byref(batch))
                assert st == 0, (st, batch.n_dropped)
                t2 = time.perf_counter()
                st = lib.jr_fsm_fold_mt(C.cast(ptr, C.c_void_p), C.c_size_t(batch.n_records), G, R, applied, totals, FOLD_THREADS)   # the host's fsm::Driver bookkeeping
                assert st == 0
                rec_bytes[0] += batch.n_records * 32 + C.sizeof(abi.FsmBatch)
                if trace is not None:
                    trace["table_wait"] += t1 - t0
                    trace["records_wait"] += t2 - t1
                    trace["fold"] += time.perf_counter() - t2

        seq = [0]      # steps submitted so far (token bases advance with it, across warm-up and timed loops)

        # JR_E2E_TWO_THREADS=1: consume on a second host thread (the engine allows it).  Measured here it is within a few percent
        # of the single-threaded loop when few threads fold and much worse when many do, so the default stays one thread.
        two_threads = os.environ.get("JR_E2E_TWO_THREADS", "0") == "1"

        def e2e_steps(n):
            """Step i is submitted by this thread and consumed (copy-out waited for, result read, Instruction records folded)
            by a second one -- josefine's Raft task and fsm::Driver task (fsm.rs:52-88).  NB staging buffers: step i + NB is
            not submitted before step i has been consumed."""
            if not two_threads:
                for j in range(min(NB - 1, n)):
                    submit(j)
                for i in range(n):
                    if i + NB - 1 < n:
                        ts = time.perf_counter()
                        submit(i + NB - 1)
                        if trace is not None:
                            trace["submit"] += time.perf_counter() - ts
                    consume(i)
                return
            free, ready, failed = threading.Semaphore(NB), threading.Semaphore(0), []

            def consumer():
                try:
                    for i in range(n):
                        ready.acquire()
                        consume(i)
                        free.release()
                except BaseException as ex:      # noqa: BLE001 -- hand it to the submitting thread
                    failed.append(ex)
                    for _ in range(n + NB):
                        free.release()

            th = threading.Thread(target=consumer, name="fsm-driver")
            th.start()
            for i in range(n):
                free.acquire()
                if failed:
                    break
                ts = time.perf_counter()
                submit(i)
                if trace is not None:
                    trace["submit"] += time.perf_counter() - ts
                ready.release()
            th.join()
            if failed:
                raise failed[0]

        e2e_steps(max(warmup, 4))
        eng.sync()
        self.barrier()
        for k in range(3):
            totals[k] = 0
        rec_bytes[0] = 0
        if trace is not None:
            for k in trace:
                trace[k] = 0.0
        t0 = time.perf_counter()
        e2e_steps(steps)
        eng.sync()
        dt = self.max_over_ranks(time.perf_counter() - t0)
        faults = eng.fault_count()
        assert faults == 0, f"{faults} replicas faulted in the end-to-end arm"
        if with_output:
            # every group-tick proposes one block; all R replicas apply it: the stream must carry ~ (R + 1) Instructions per group-tick
            expect = G * S * steps * (R + 1)
            got = int(totals[0] + totals[1])
            assert abs(got - expect) <= expect * 0.02 + 4 * G * R, (got, expect)
        out = {"value": self.world * G * S * steps / dt, "unit": UNIT, "h2d_bytes_per_step": S * G * 8 if dense_input else G * 16,
               "folded_groups_last_step": eng.fold_count(),
               "input": "dense: one u64 token per group-tick (jr_run_tokens)" if dense_input else
                        "run-length: one {base, stride} per group and step (jr_run_token_runs); the same tokens",
               "d2h_bytes_per_step": G * 16 + (rec_bytes[0] // steps if with_output else 0), "ms_per_step": dt * 1e3 / steps,
               "commit_last": checks[-1], "faulted_replicas": faults,
               "timing": "host wall clock around all timed steps incl. the final sync, max over ranks",
               "l2": "steps run back to back, no flush in between: one step moves ~0.4 GB through DRAM (profiles/, ncu), more than the 126 MB L2"}
        if trace is not None:
            out["host_ms_per_step"] = {k: v * 1e3 / steps for k, v in trace.items()}      # timed steps only
        if with_output:
            out.update({"instructions_per_step": int(totals[0] + totals[1]) // steps, "records_per_step": int(totals[2]) // steps,
                        "d2h_stream_bytes_per_step": rec_bytes[0] // steps,
                        "api": "per step: " + ("jr_run_tokens(pinned u64 tokens[64][G]" if dense_input else "jr_run_token_runs(pinned jr_token_run[G]") +
                               ", routed to the last announced leader; ends with jr_truncate: jr_set_auto_truncate) + "
                               "jr_leader_table_async(pinned jr_leader_entry[G]) + jr_fsm_records_async; then jr_leader_table_wait + "
                               f"jr_fsm_records_wait + jr_fsm_fold_mt over the batch on {FOLD_THREADS} host threads (apply watermark per replica), "
                               + ("on a second host thread (the fsm::Driver task); " if two_threads else "") + f"{NB} steps in flight",
                        "host_fold_threads": FOLD_THREADS})
        else:
            out["api"] = ("per step: jr_run_tokens (ends with jr_truncate) + jr_leader_table_async + jr_leader_table_wait; engine created without "
                          "JR_F_CAPTURE_FSM (round 1's end-to-end leg)")
        del eng
        torch.cuda.empty_cache()
        return out

    # ---- BASELINE config #2: 1,024 x 3, cold start -> elections -> 64 proposals -> 256 ticks in all
    def config2(self, reps):
        torch = self.torch
        G, R = 1024, 3
        eng = self.make(G, R, seed=0, chain_capacity=256, flags=abi.F_CAPTURE_FSM, fsm_units=64)
        eng.set_stream(self.stream.cuda_stream)
        per = []
        for rep in range(reps + 2):
            eng.reset()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(self.stream)
            eng.run(DT_MS, DT_MS, 100, 0)              # cold start: seeded timeouts, one election per group
            eng.run(DT_MS * 101, DT_MS, 64, 1)         # 64 client proposals per group
            eng.run(DT_MS * 165, DT_MS, 92, 0)
            b.record(self.stream)
            torch.cuda.synchronize()
            if rep >= 2:
                per.append(a.elapsed_time(b))
            eng.discard_fsm(strict=False)
        leaders = sum(1 for (_, l, _) in eng.leader_table() if l)
        ms = statistics.median(per)
        return {"workload": "BASELINE config #2: 1,024 groups x 3 replicas, cold start -> seeded timeouts -> elections -> 64 client "
                            "proposals/group, 256 ticks (3 fused launches)", "groups": G, "replicas": R, "ticks": 256,
                "ms_per_trace": ms, "value": G * 256 / (ms * 1e-3), "unit": UNIT, "groups_with_leader": leaders,
                "faulted_replicas": eng.fault_count(),
                "note": "32 CTAs on 148 SMs: this size measures launch + per-tick latency, not throughput"}

    # ---- BASELINE config #5: 65,536 x 7, 10% of the groups lose their leader every 100 ticks, compact every 256
    def config5(self, steps, warmup):
        torch = self.torch
        G, R, S = GROUPS_PER_GPU, 7, TICKS_PER_STEP
        eng = self.steady_engine(G, R, abi.F_CAPTURE_FSM, seed=2, auto_truncate=False)    # several runs per step here: one explicit jr_truncate at its end
        tick = [16]
        now = lambda: DT_MS * (tick[0] + 1)   # noqa: E731
        compact_ev, kills = [], []

        def one_step():
            left = S
            while left:
                to_kill = 100 - tick[0] % 100
                to_compact = 256 - tick[0] % 256
                n = min(left, to_kill, to_compact)
                eng.run(now(), DT_MS, n, 1)
                tick[0] += n
                left -= n
                if tick[0] % 100 == 0:
                    kills.append(eng.kill_leaders(tick[0], 100))
                if tick[0] % 256 == 0:
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(self.stream)
                    eng.compact()
                    b.record(self.stream)
                    compact_ev.append((a, b))
            eng.truncate(TRUNC_MARGIN)
            eng._lib.jr_fsm_records_async(eng._h)
            ptr, batch = C.POINTER(abi.FsmRecord)(), abi.FsmBatch()
            assert eng._lib.jr_fsm_records_wait(eng._h, C.byref(ptr), C.byref(batch)) == 0

        for _ in range(warmup):
            one_step()
        torch.cuda.synchronize()
        compact_ev.clear()
        evs = []
        for _ in range(steps):
            self.flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(self.stream)
            one_step()
            b.record(self.stream)
            evs.append((a, b))
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        table = eng.leader_table()
        live = sum(1 for (_, l, _) in table if l)
        st = eng.query_many([(g, 1 + (g % R)) for g in range(0, G, 257)])
        span = statistics.mean(max(int(s.commit) - int(s.chain_floor), 0) for s in st)
        cms = statistics.median(a.elapsed_time(b) for a, b in compact_ev) if compact_ev else None
        cbytes = 4 * span * R * G
        faults = eng.fault_count()
        res = {"workload": "BASELINE config #5: 65,536 groups x 7 replicas, 1 proposal/group/tick, the leader of 10% of the groups "
                           "(counter RNG) silenced every 100 ticks, Chain::compact on every replica every 256 ticks, jr_truncate every 64",
               "groups": G, "replicas": R, "ticks_per_step": S, "steps": steps, "ms_per_step": ms / steps,
               "value": G * S * steps / (ms * 1e-3), "unit": UNIT, "groups_with_live_leader_at_end": live,
               "leaders_silenced": int(sum(kills)), "faulted_replicas": faults,
               "compact_kernel": {"ms": cms, "launches": len(compact_ev), "bytes": cbytes,
                                  "gbs": (cbytes / (cms * 1e-3) / 1e9) if cms else None,
                                  "note": "walks ids [floor, commit) of every replica: 4 B x (commit - floor) x R x G; the window is "
                                          f"~{span:.0f} ids because jr_truncate runs every step"},
               "note": "SURVEY N1: a follower that ever heard a heartbeat keeps voted_for = the silenced leader and never starts an "
                       "election, so silenced groups stay leaderless (reference behaviour, reproduced); the live fraction decays"}
        del eng
        torch.cuda.empty_cache()
        return res

    # ---- digest parity against the C++ restatement, same inputs, in this run
    def parity(self, name, G, R, seed, ticks=TICKS_PER_STEP, kind="steady"):
        fl = abi.F_STREAM_DIGEST
        e = self.make(G, R, seed=seed, chain_capacity=CHAIN_WINDOW, flags=fl, fsm_units=FSM_UNITS)
        e.set_stream(self.stream.cuda_stream)
        from oracle.restated import RestatedCluster
        threads = best_cpu_threads(R, effective_cores())
        o = RestatedCluster.create(G, R, n_threads=threads, seed=seed, chain_capacity=CHAIN_WINDOW, flags=fl)
        t0 = time.perf_counter()
        for api in (e, o):
            if kind == "cold":             # config #2's trace: cold start, elections, 64 proposals, 256 ticks
                api.run(DT_MS, DT_MS, 100, 0)
                api.run(DT_MS * 101, DT_MS, 64, 1)
                api.run(DT_MS * 165, DT_MS, 92, 0)
                continue
            api.step(0, flags=0, inject=bootstrap_inject(G, R))
            api.run(DT_MS, DT_MS, ticks // 2, 1)
            if kind == "churn":
                api.kill_leaders(50, 100)
                api.compact()
            api.truncate(TRUNC_MARGIN)
            api.run(DT_MS * (ticks // 2 + 1), DT_MS, ticks - ticks // 2, 1)
        ok = (e.state_digest() == o.state_digest() and e.stream_digest() == o.stream_digest()
              and e.fault_count() == o.fault_count() and e.leader_table() == o.leader_table())
        res = {"config": name, "groups": G, "replicas": R, "ticks": ticks, "bit_exact": bool(ok),
               "checked": "state digest (all replica state + block tables), Message and Instruction stream digests, fault count, "
                          "leader table", "against": "C++ restatement of josefine src/raft (oracle/)", "seconds": time.perf_counter() - t0}
        del e, o
        self.torch.cuda.empty_cache()
        return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--groups", type=int, default=GROUPS_PER_GPU, help="groups per GPU")
    ap.add_argument("--replicas", type=int, default=REPLICAS)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip configs #2/#4/#5 and the variants")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the headline arm's last timed step returned (its Instruction-record batch and the "
                         "leader table after it; rank 0's shard) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    bn = Bench(args)
    world, rank = bn.world, bn.rank
    G, R, S = args.groups, args.replicas, TICKS_PER_STEP
    sampler = ClockSampler(bn.local) if rank == 0 else None
    if sampler:
        sampler.start()

    # ---------------- headline: config #3, device resident ----------------
    main_res = bn.device_resident(G, R, args.steps, max(args.warmup, 20), sampler=sampler,   # >= 20 untimed steps: also nvidia-smi's start-up
                                  keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, main_res.pop("outputs"))
    clocks = main_res.pop("clocks")
    value, ms = main_res["value"], main_res["ms_total"]
    launches = args.steps * (6 + (1 if world > 1 else 0))   # sym2_kernel, step_kernel, truncate_kernel, fsm count / scan / pack (+ leader_table_kernel); the copy-out is a DMA

    # ---------------- end to end ----------------
    e2e = e2e_plain = e2e_dense = None
    if not args.no_e2e:
        e2e = bn.end_to_end(G, R, args.steps, args.warmup, with_output=True)
        e2e_dense = bn.end_to_end(G, R, args.steps, args.warmup, with_output=True, dense_input=True)
        e2e_plain = bn.end_to_end(G, R, args.steps, args.warmup, with_output=False, dense_input=True)

    # ---------------- other BASELINE configs, variants ----------------
    others, variants = {}, {}
    short = max(20, args.steps // 4)
    if not args.no_others:
        r4 = bn.device_resident(2 * GROUPS_PER_GPU, 5, short, 5)
        others["config4_shard"] = {
            "workload": f"BASELINE config #4: 1,048,576 groups x 5 replicas over 8 GPUs = 131,072 per GPU; here {world} GPU(s) x 131,072 "
                        f"= {world * 2 * GROUPS_PER_GPU} groups, leader announce all-gathered every step" + ("" if world > 1 else " (no peer at N=1)"),
            "groups_per_gpu": 2 * GROUPS_PER_GPU, "replicas": 5, "steps": short, "ms_per_step": r4["ms_per_step"], "value": r4["value"],
            "unit": UNIT, "faulted_replicas": r4["faulted_replicas"], "collective_us": r4["collective_us"]}
        v1 = bn.device_resident(G, R, short, 5, announce=False, scattered=True)
        variants["scattered_leaders"] = {"value": v1["value"], "ms_per_step": v1["ms_per_step"],
                                         "what": "leader of group g on node g % R + 1 (what real elections leave behind) instead of node 1"}
        v2 = bn.device_resident(G, R, short, 5, announce=False, heartbeat_ms=99)
        variants["heartbeat_every_tick"] = {"value": v2["value"], "ms_per_step": v2["ms_per_step"],
                                            "what": "heartbeat_ms = 99 < tick: the leader heartbeats every tick (a wall-clock josefine does), not every second one"}
        if rank == 0:
            others["config2"] = bn.config2(8)
            others["config5"] = bn.config5(short, 4)
        bn.barrier()

    if rank != 0:
        if world > 1:
            bn.dist.destroy_process_group()
        return

    parity = []
    if not args.no_parity and world == 1:
        parity.append(bn.parity("#3 65,536x5 steady", GROUPS_PER_GPU, 5, SEED))
        if not args.no_others:
            parity.append(bn.parity("#2 1,024x3 cold start", 1024, 3, 0, ticks=256, kind="cold"))
            parity.append(bn.parity("#4 shard 131,072x5", 2 * GROUPS_PER_GPU, 5, SEED, ticks=32))
            parity.append(bn.parity("#5 65,536x7 churn+compact", GROUPS_PER_GPU, 7, 2, ticks=48, kind="churn"))
        assert all(p["bit_exact"] for p in parity), parity

    # ---------------- roofline + cpu baseline (rank 0) ----------------
    ref_bytes, lay_bytes = algorithmic_bytes_per_group_tick(bn.make, R)
    peak, peak_src = measured_peak()
    avg_launch_s = (ms * 1e-3) / args.steps            # one step = S fused ticks of all G groups
    traffic, kernel_s = None, None
    kernel_name = f"step_kernel<{R}>"
    for name in ("dominant_kernel_latest.json", "step_kernel_latest.json"):
        prof = os.path.join(ROOT, "profiles", name)
        if os.path.exists(prof):   # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this
            pj = json.load(open(prof))       # command, per launch (one launch = TICKS_PER_STEP ticks)
            if pj.get("ticks_per_launch") == S and pj.get("groups") == G:
                traffic = pj["dram_bytes_per_launch"]
                kernel_name = pj["kernel"].split("(")[0].replace("void ", "")
                kernel_s = pj["duration_s"]
                break
    ach_ref = ref_bytes * G * S / avg_launch_s / 1e9
    ach_lay = lay_bytes * G * S / avg_launch_s / 1e9
    roofline = {"bound": "hbm", "achieved": ach_ref, "peak": peak, "unit": "GB/s", "frac": ach_ref / peak,
                "frac_reference_widths": ach_ref / peak, "frac_layout": ach_lay / peak,
                "frac_dram": (traffic / kernel_s / 1e9 / peak) if traffic else None,
                "traffic": traffic, "kernel": kernel_name, "algorithmic_bytes_per_group_tick": ref_bytes,
                "layout_bytes_per_group_tick": lay_bytes, "avg_launch_us": avg_launch_s * 1e6, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": ref_bytes * G * S,
                "note": f"`frac` counts the bytes a group-tick moves in the REFERENCE's widths (SURVEY 8d formula applied to this workload's "
                        f"measured message mix, heartbeat every second tick); frac_layout uses this engine's wider units and is not the claim; "
                        f"frac_dram is the real DRAM traffic of the dominant kernel (profiles/dominant_kernel_latest.json) over its own duration.  One launch = {S} fused ticks of {G} groups with "
                        f"state in registers and mailboxes in shared memory, so most algorithmic bytes never reach DRAM: the kernel is latency "
                        f"bound, not bandwidth bound (DESIGN.md section 6)."}
    cpu = None
    if not args.no_cpu and world == 1:
        cpu = cpu_baseline_block(G, R)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(G, R),
                   "groups_per_gpu": G, "replicas": R, "ticks_per_step": S, "tick_ms": DT_MS, "seed": SEED,
                   "heartbeat": "heartbeat_ms = tick = 100 and a strict `>` (leader.rs:78-84): every second tick",
                   "chain_window": CHAIN_WINDOW, "truncate": f"jr_truncate(margin {TRUNC_MARGIN}) at the end of every fused run (jr_set_auto_truncate), inside the timed region (D7); no engine reset",
                   "output": "Instruction stream drained every step (jr_fsm_records_async), folded on the host one step later",
                   "l2": f"flushed between timed steps ({L2_FLUSH_BYTES >> 20} MiB write); ticks inside a step run back to back",
                   "parallelism": f"groups sharded over {world} GPU(s); leader-announce all_gather once per step" if world > 1
                   else "single GPU", "faulted_replicas": main_res["faulted_replicas"], "commit_min": main_res["commit_min"],
                   "untimed_steps_before_timing": max(args.warmup, 20), "host_placement": bn.placement},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_dense_input": e2e_dense, "e2e_no_output": e2e_plain, "gpu_launches": launches, "clocks": clocks,
        "collective_us": main_res["collective_us"], "instructions_per_step": main_res["instructions"] // args.steps,
        "other_configs": others, "variants": variants, "parity": parity,
    }
    print(json.dumps(line))
    if world > 1:
        bn.dist.destroy_process_group()


if __name__ == "__main__":
    main()
