"""The symmetric-group fold (josefine_b200/csrc/sym_fold.cuh): jr_run* applies a whole launch of a symmetric group in
two lanes of sym2_kernel, one for the leader and one standing for every follower.  It must be indistinguishable from
step_kernel: replica state, block tables, leader tables and Instruction streams equal those of an engine that never
folds (JR_F_NO_SYMMETRIC_FOLD) AND those of the oracle.  (Engines with JR_F_STREAM_DIGEST never fold, so the
digest-based parity suites keep testing step_kernel; here everything except the Message stream is compared.)"""
import pytest

from josefine_b200 import abi, Command, fsm_tuple
from tests import parity
from tests.stream_cases import _bootstrap, strided_tokens

CAP = abi.F_CAPTURE_FSM


def _oracle(g, r, **kw):
    from oracle.restated import RestatedCluster
    return RestatedCluster.create(g, r, **kw)


def _emu(g, r, **kw):
    from tests.emu.emu import EmuEngine
    return EmuEngine.create(g, r, **kw)


def _gpu(g, r, **kw):
    from josefine_b200 import RaftEngine
    return RaftEngine.create(g, r, **kw)


def trio(make, G, R, **cfg):
    cfg.setdefault("flags", CAP)
    fold = make(G, R, **cfg)
    plain = make(G, R, **dict(cfg, flags=cfg["flags"] | abi.F_NO_SYMMETRIC_FOLD))
    ora = _oracle(G, R, **cfg)
    return fold, plain, ora


def same(apis, chain_ids=48, fsm_cap=None):
    a = apis[0]
    fsm_cap = fsm_cap or max(1 << 16, a.n_groups * a.n_replicas * 160)
    streams = [[fsm_tuple(f) for f in api.drain_fsm(cap=fsm_cap)] for api in apis]
    for other, st in zip(apis[1:], streams[1:]):
        assert streams[0] == st, "Instruction streams differ"
        parity.compare_states(a, other, chain_ids=chain_ids)
        assert a.state_digest() == other.state_digest()
        assert a.leader_table() == other.leader_table()
        assert a.fault_count() == other.fault_count()


def case_steady(make, R, G=40, hb=100, dt=100, launches=5, ticks=33, n_synth=1):
    apis = trio(make, G, R, seed=R, heartbeat_ms=hb, chain_capacity=512, fsm_units=256)
    for api in apis:
        _bootstrap(api, G, R)
    now = dt
    folded = []
    for k in range(launches):
        for api in apis:
            api.run(now, dt, ticks, n_synth)
        now += dt * ticks
        folded.append(apis[0].fold_count())
        assert apis[1].fold_count() == 0
        same(apis)
    return folded


def case_tokens_kill_truncate(make, G=48, R=5):
    """jr_run_tokens (routed proposals, some ticks without one), leaders silenced in between (those groups leave the fold),
    jr_truncate moving the window under it."""
    apis = trio(make, G, R, seed=9, chain_capacity=128, fsm_units=64, fsm_host_records=G * R * 32)   # holes in the token grid: short runs
    for api in apis:
        _bootstrap(api, G, R)
        api.run(100, 100, 12, 1)
        api.leader_table()
    now, tick = 1300, 0
    folded = []
    for rnd in range(6):
        toks = strided_tokens(20, G, tick)
        for k in range(20):
            if (k + rnd) % 7 == 3:
                toks[k] = [0] * G                       # a tick without proposals
        for api in apis:
            api.run_tokens(now, 100, toks)
            api.truncate(6)
        now += 2000
        tick += 20
        folded.append(apis[0].fold_count())
        same(apis, chain_ids=0)
        if rnd == 2:
            assert len({api.kill_leaders(4, 300) for api in apis}) == 1
        if rnd == 3:
            for api in apis:
                api.leader_table()                      # re-announce: dead groups now drop their tokens
    reqs = [(g, n, max(int(apis[0].query(g, n).chain_floor), 0), 40) for g in range(0, G, 7) for n in (1, 2)]
    assert apis[0].chain_read_many(reqs) == apis[1].chain_read_many(reqs) == apis[2].chain_read_many(reqs)
    return folded


def case_auto_truncate(make, G=96, R=5):
    """jr_set_auto_truncate: a fused run that ends with its own truncation (done by the folding lane for folded groups,
    by truncate_kernel for the rest) equals run + jr_truncate on a non-folding engine and on the oracle -- and the
    oracle's own auto mode equals its explicit calls.  Some leaders are silenced on the way so both paths are taken."""
    cfg = dict(seed=11, chain_capacity=128, fsm_units=128, fsm_host_records=G * R * 32)
    apis = trio(make, G, R, **cfg)
    ora_auto = _oracle(G, R, flags=CAP, **cfg)
    apis = list(apis) + [ora_auto]
    for api in apis:
        _bootstrap(api, G, R)
        api.run(100, 100, 12, 1)
    apis[0].set_auto_truncate(5)
    ora_auto.set_auto_truncate(5)
    now = 1300
    folded = []
    for rnd in range(6):
        ticks = 17 + 3 * rnd
        for i, api in enumerate(apis):
            api.run(now, 100, ticks, 1)
            if i in (1, 2):
                api.truncate(5)
        now += 100 * ticks
        folded.append(apis[0].fold_count())
        same(apis, chain_ids=0)
        if rnd == 2:
            assert len({api.kill_leaders(8, 250) for api in apis}) == 1
    floors = [int(apis[0].query(g, 1).chain_floor) for g in range(0, G, 5)]
    assert max(floors) > 60                                       # the window really moved
    apis[0].set_auto_truncate(None)
    ora_auto.set_auto_truncate(None)
    for i, api in enumerate(apis):
        api.run(now, 100, 9, 1)                                   # switched off again: floors stay
    assert [int(apis[0].query(g, 1).chain_floor) for g in range(0, G, 5)] == floors
    same(apis, chain_ids=0)
    return folded


def case_misrouted_and_asymmetric(make, G=16, R=3):
    """Groups that must NOT fold: a proposal aimed at a follower (proxied ClientRequest), a follower silenced (asymmetric),
    elections in progress.  Everything still equals the oracle, the eligible rest folds."""
    apis = trio(make, G, R, seed=4, chain_capacity=256, fsm_units=128)
    for api in apis:
        _bootstrap(api, G, R)
        api.run(100, 100, 10, 1)
        api.set_alive(3, 2, False)                      # group 3 loses a follower
    props = [[((2 if g == 5 else 1), 7000 + 100 * k + g) for g in range(G)] for k in range(12)]   # group 5: proposals to follower 2
    for api in apis:
        api.run_proposals(1100, 100, props)
    n = apis[0].fold_count()
    same(apis)
    for api in apis:
        api.run(2300, 100, 15, 1)         # group 5 still has proxied mail in flight when this launch starts
    same(apis)
    for api in apis:
        api.run(3800, 100, 15, 1)
    same(apis)
    return n, apis[0].fold_count()


@pytest.mark.parametrize("R", [2, 3, 5, 7])
def test_steady_fold_on_device_code(R):
    folded = case_steady(_emu, R)
    assert folded[0] == 0 and all(f == 40 for f in folded[1:]), folded   # first launch starts from the election's mail: not canonical


@pytest.mark.parametrize("hb,dt", [(99, 100), (100, 50), (250, 100), (100, 100)])
def test_heartbeat_cadences_on_device_code(hb, dt):
    folded = case_steady(_emu, 5, G=8, hb=hb, dt=dt, launches=4, ticks=21)
    assert folded[-1] == 8, folded


def test_no_proposals_and_two_per_tick_on_device_code():
    assert case_steady(_emu, 5, G=8, n_synth=0)[-1] == 8
    assert case_steady(_emu, 3, G=8, n_synth=2)[-1] == 8


def test_tokens_kill_truncate_on_device_code():
    folded = case_tokens_kill_truncate(_emu)
    assert folded[1] == 48 and 0 < folded[-1] < 48, folded


def test_auto_truncate_on_device_code():
    folded = case_auto_truncate(_emu)
    assert folded[0] == 96 and 0 < folded[-1] < 96


def test_misrouted_and_asymmetric_on_device_code():
    n1, n2 = case_misrouted_and_asymmetric(_emu)
    assert n1 == 16 - 2 and n2 == 16 - 1, (n1, n2)      # groups 3 and 5 stay out; group 5 comes back once proposals go to the leader


def test_split_launches_with_fold_on_device_code(monkeypatch):
    monkeypatch.setenv("JR_PARTS", "3")
    assert case_steady(_emu, 3, G=70, launches=3, ticks=25)[-1] == 70


@pytest.mark.gpu
@pytest.mark.parametrize("R", [3, 5, 7])
def test_steady_fold_on_gpu(R):
    folded = case_steady(_gpu, R, G=3000, launches=4, ticks=40)
    assert all(f == 3000 for f in folded[1:]), folded


@pytest.mark.gpu
def test_tokens_kill_truncate_on_gpu():
    case_tokens_kill_truncate(_gpu, G=2048)


@pytest.mark.gpu
def test_auto_truncate_on_gpu():
    folded = case_auto_truncate(_gpu, G=4096)
    assert folded[0] == 4096 and 0 < folded[-1] < 4096


@pytest.mark.gpu
def test_misrouted_and_asymmetric_on_gpu():
    case_misrouted_and_asymmetric(_gpu)


def case_token_runs_equal_tokens(make, G=24, R=5):
    """jr_run_token_runs(base, stride) == jr_run_tokens(base + k * stride), folded or not, and on the oracle."""
    fold, plain, ora = trio(make, G, R, seed=6, chain_capacity=256, fsm_units=64)
    ref = make(G, R, seed=6, chain_capacity=256, fsm_units=64, flags=CAP)
    for api in (fold, plain, ora, ref):
        _bootstrap(api, G, R)
        api.run(100, 100, 12, 1)
        api.leader_table()
    now = 1300
    for rnd in range(3):
        runs = [(0, 0) if (g + rnd) % 6 == 0 else (((rnd + 1) << 40) + g + 1, 1 << 20) for g in range(G)]
        n = 17 + rnd
        for api in (fold, plain, ora):
            api.run_token_runs(now, 100, n, runs)
        ref.run_tokens(now, 100, [[(b + k * s) if b else 0 for (b, s) in runs] for k in range(n)])
        now += 100 * n
        same([fold, plain, ora, ref])
    return fold.fold_count()


def test_token_runs_on_device_code():
    assert case_token_runs_equal_tokens(_emu) == 24


@pytest.mark.gpu
def test_token_runs_on_gpu():
    assert case_token_runs_equal_tokens(_gpu, G=1500) == 1500


# ---------------------------------------------------------------------------------------------------------------------
# Randomised scripts: every launch shape the fused calls have, with faults, silenced and revived nodes, proposals aimed at
# followers, holes in the token grid, truncation (explicit and fused) and compaction thrown in -- so groups enter the
# fold, abort out of it in the middle of a launch (either lane of sym2_kernel first), fall back to step_kernel and come
# back.  After every launch the folding engine, the never-folding engine and the oracle must agree on everything.

def _random_script(make, seed, rounds=9, **cfg_over):
    import random
    rng = random.Random(seed)
    G, R = rng.choice([(40, 3), (64, 5), (33, 5), (24, 7)])
    cfg = dict(seed=seed, chain_capacity=512, fsm_units=512, fsm_host_records=G * R * 1024,
               heartbeat_ms=rng.choice([100, 100, 99, 250]), mailbox_units=64)
    cfg.update(cfg_over)
    apis = trio(make, G, R, **cfg)
    lead = rng.choice([1, 2]) if seed % 3 else 1
    for api in apis:
        _bootstrap(api, G, R, node=lead)
        api.run(100, 100, 10, 1)
        api.leader_table()
    now, tick = 1100, 0
    auto = None
    folded_any = unfolded_any = False
    for rnd in range(rounds):
        kind = rng.choice(["run", "run", "tokens", "token_runs", "proposals"])
        ticks = rng.choice([2, 3, 7, 16, 21, 33])
        if rng.random() < 0.25:                              # switch the fused truncation on / off / to another margin
            auto = rng.choice([None, 3, 6, 9])
            for api in apis:
                api.set_auto_truncate(auto)
        if kind == "run":
            n_synth = rng.choice([0, 1, 1, 2])
            for api in apis:
                api.run(now, 100, ticks, n_synth)
        elif kind == "tokens":
            toks = strided_tokens(ticks, G, tick)
            for k in range(ticks):
                if rng.random() < 0.2:
                    toks[k] = [0] * G                        # a tick without proposals
                elif rng.random() < 0.2:
                    toks[k] = [t if rng.random() < 0.7 else 0 for t in toks[k]]   # holes
            for api in apis:
                api.run_tokens(now, 100, toks)
        elif kind == "token_runs":
            runs = [(((rnd + 1) << 44) + g + 1 if rng.random() < 0.9 else 0, rng.choice([1, 1 << 20, 1 << 32])) for g in range(G)]
            for api in apis:
                api.run_token_runs(now, 100, ticks, runs)
        else:                                                # dense proposals, some aimed at followers / nobody
            props = [[(rng.choice([1, 1, 1, 2, 0, R]) if rng.random() < 0.15 else 1, 9000 + 1000 * rnd + 37 * k + g) for g in range(G)]
                     for k in range(ticks)]
            for api in apis:
                api.run_proposals(now, 100, props)
        now += 100 * ticks
        tick += ticks
        n = apis[0].fold_count()
        folded_any |= n > 0
        unfolded_any |= n < G
        assert apis[1].fold_count() == 0
        if auto is None and rng.random() < 0.5:
            m = rng.choice([2, 5, 8])
            for api in apis:
                api.truncate(m)
        same(apis, chain_ids=0)
        r = rng.random()
        if r < 0.2:
            permille = rng.choice([100, 300])
            assert len({api.kill_leaders(seed * 31 + rnd, permille) for api in apis}) == 1
        elif r < 0.4:
            g, node, alive = rng.randrange(G), rng.randrange(1, R + 1), rng.random() < 0.4
            for api in apis:
                api.set_alive(g, node, alive)
        elif r < 0.5:
            for api in apis:
                api.compact()
        if rng.random() < 0.5:
            for api in apis:
                api.leader_table()                           # re-announce: routes follow the (possibly silenced) leaders
    reqs = [(g, n, max(int(apis[0].query(g, n).chain_floor), 0), 24) for g in range(0, G, 5) for n in (1, R)]
    assert apis[0].chain_read_many(reqs) == apis[1].chain_read_many(reqs) == apis[2].chain_read_many(reqs)
    return folded_any, unfolded_any


@pytest.mark.parametrize("seed", range(12))
def test_random_scripts_on_device_code(seed):
    folded_any, _ = _random_script(_emu, seed)
    assert folded_any


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [100, 101, 102, 103])
def test_random_scripts_on_gpu(seed):
    folded_any, _ = _random_script(_gpu, seed, rounds=12)
    assert folded_any
