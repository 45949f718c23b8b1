#!/usr/bin/env python
"""Small fused-kernel workload for compute-sanitizer (memcheck / racecheck / synccheck):
cold-start elections at R=3, bootstrapped steady state at R=5 and R=7 with tiny
shared-memory mailboxes (spill path), compact, kill_leaders, inject + capture."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from josefine_b200 import abi, RaftEngine  # noqa: E402
from tests.golden_scenarios import bootstrap  # noqa: E402

for R, G in ((3, 70), (5, 64), (7, 33)):
    e = RaftEngine.create(G, R, seed=R, flags=abi.F_CAPTURE_MESSAGES | abi.F_CAPTURE_FSM | abi.F_STREAM_DIGEST,
                          chain_capacity=128, fsm_units=128)
    if R == 3:
        e.run(100, 100, 40, 1)
    else:
        e.step(0, flags=0, inject=bootstrap(G, R))
        e.run(100, 100, 24, 1)
    e.step(9000, n_synth=1)
    e.kill_leaders(1, 300)
    e.compact()
    e.run(9100, 100, 8, 1)
    print(R, e.state_digest(), e.fault_count(), e.stream_digest()[2:])
print("sanitize workload done")

# round 2: the symmetric-group fold, the Instruction-stream drain, truncation, restart, bulk introspection, checkpoint
for R, G in ((3, 70), (5, 96)):
    e = RaftEngine.create(G, R, seed=R, flags=abi.F_CAPTURE_FSM, chain_capacity=64, fsm_units=32)
    e.step(0, flags=0, inject=bootstrap(G, R))
    folded = []
    now = 100
    for rnd in range(6):
        if rnd == 4:
            e.set_auto_truncate(4)          # the fold truncates its groups itself from here on (sym2_kernel's tail)
        e.run(now, 100, 20, 1)
        now += 2000
        folded.append(e.fold_count())
        if rnd < 4:
            e.truncate(4)
        recs, batch = e.fsm_records()
        assert batch.n_dropped == 0 and len(e.fsm_expand(recs)) == batch.n_instructions
        if rnd == 2:
            e.kill_leaders(3, 200)
            e.leader_table()
        if rnd >= 3:
            e.run_token_runs(now, 100, 10, [((rnd << 40) + g + 1, 1 << 20) for g in range(G)])
            now += 1000
    blob = e.save()
    e.restore(blob)
    st = e.query_many([(g, 1 + g % R) for g in range(G)])
    e.chain_read_many([(g, 1, int(st[g].chain_floor), 8) for g in range(0, G, 9)])
    blocks = [b for b in e.chain_read(0, 2, int(st[0].chain_floor), 40) if b is not None]
    e.node_restart(0, 2, now, blocks, int(e.query(0, 2).commit))
    e.run(now, 100, 6, 1)
    print(R, "folded per launch", folded, e.state_digest(), e.fault_count())
print("round-2 sanitize workload done")
