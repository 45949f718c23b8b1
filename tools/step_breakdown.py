#!/usr/bin/env python
"""Where one bench step's device time goes: CUDA events between the three calls of a step (fused run, truncate, drain)
on the engine's stream, for the headline workload and its variants.  Diagnostic; bench.py holds the reported numbers.

usage: step_breakdown.py [steps]"""
import argparse
import ctypes as C
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from josefine_b200 import abi  # noqa: E402


EXPLICIT_TRUNCATE = False


def measure(bn, label, G, R, steps, capture=True, flush=True, fold=True, **kw):
    torch = bn.torch
    flags = (abi.F_CAPTURE_FSM if capture else 0) | (0 if fold else abi.F_NO_SYMMETRIC_FOLD)
    eng = bn.steady_engine(G, R, flags, auto_truncate=not EXPLICIT_TRUNCATE, **kw)
    lib, h = eng._lib, eng._h
    S = bench.TICKS_PER_STEP
    now = bench.DT_MS * 17
    outstanding = 0
    segs = {"run": [], "truncate": [], "drain": [], "step": []}

    def take():
        ptr, batch = C.POINTER(abi.FsmRecord)(), abi.FsmBatch()
        assert lib.jr_fsm_records_wait(h, C.byref(ptr), C.byref(batch)) == 0

    for i in range(steps + 5):
        if flush:
            bn.flush.fill_(1)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record(bn.stream)
        eng.run(now, bench.DT_MS, S, 1)          # ends with its own truncation (jr_set_auto_truncate) unless --explicit-truncate
        ev[1].record(bn.stream)
        if EXPLICIT_TRUNCATE:
            eng.truncate(bench.TRUNC_MARGIN)
        ev[2].record(bn.stream)
        if capture:
            assert lib.jr_fsm_records_async(h) == 0
            outstanding += 1
        ev[3].record(bn.stream)
        if outstanding == 2:
            take()
            outstanding -= 1
        now += bench.DT_MS * S
        if i >= 5:
            segs["_ev"] = segs.get("_ev", []) + [ev]
    while outstanding:
        take()
        outstanding -= 1
    torch.cuda.synchronize()
    for ev in segs.pop("_ev"):
        segs["run"].append(ev[0].elapsed_time(ev[1]))
        segs["truncate"].append(ev[1].elapsed_time(ev[2]))
        segs["drain"].append(ev[2].elapsed_time(ev[3]))
        segs["step"].append(ev[0].elapsed_time(ev[3]))
    out = {k: round(statistics.mean(v) * 1e3, 1) for k, v in segs.items()}
    print(f"{label:34s} us/step {out}  folded {eng.fold_count()}/{G}  faults {eng.fault_count()}", flush=True)
    del eng
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("steps", nargs="?", type=int, default=60)
    ap.add_argument("--only", type=int, default=99, help="run only the first N variants")
    ap.add_argument("--explicit-truncate", action="store_true", help="jr_truncate as its own call (the pre-fusion shape)")
    a = ap.parse_args()
    global EXPLICIT_TRUNCATE
    EXPLICIT_TRUNCATE = a.explicit_truncate
    bn = bench.Bench(argparse.Namespace())
    G, R = bench.GROUPS_PER_GPU, bench.REPLICAS
    variants = [("headline", G, {}), ("headline, no capture", G, {"capture": False}), ("scattered leaders", G, {"scattered": True}),
                ("headline, warm L2 (no flush)", G, {"flush": False}), ("heartbeat every tick", G, {"heartbeat_ms": 99}),
                ("131,072 groups", 2 * G, {}), ("headline, fold off (step_kernel)", G, {"fold": False}),
                ("no capture, fold off", G, {"capture": False, "fold": False})]
    for label, g, kw in variants[:a.only]:
        measure(bn, label, g, R, a.steps, **kw)


if __name__ == "__main__":
    main()
