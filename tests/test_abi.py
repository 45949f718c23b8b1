"""CPU: the C-ABI library builds, loads and exports every symbol the header declares
(no compute calls -- there is no GPU here), and the ctypes mirror matches the header."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest

from josefine_b200 import abi
from josefine_b200.raft import ENGINE_LIB_PATH

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "josefine_raft_abi.h")


@pytest.fixture(scope="module")
def engine_lib():
    if not os.path.exists(ENGINE_LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return C.CDLL(ENGINE_LIB_PATH)


def test_header_symbols_match_python_list():
    text = open(HEADER).read()
    declared = set(re.findall(r"^\s*(?:jr_status|void|const char\*|uint32_t)\s+(jr_\w+)\s*\(", text, re.M))
    assert declared == set(abi.ENGINE_SYMBOLS)


def test_library_exports_every_declared_symbol(engine_lib):
    for name in abi.ENGINE_SYMBOLS:
        assert hasattr(engine_lib, name), name


def test_struct_sizes_match_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "josefine_raft_abi.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n",'
                   "sizeof(jr_config),sizeof(jr_block),sizeof(jr_msg),sizeof(jr_fsm_instr),sizeof(jr_proposal),"
                   "sizeof(jr_leader_entry),sizeof(jr_step_args),sizeof(jr_replica_state));return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [C.sizeof(t) for t in (abi.Config, abi.Block, abi.Msg, abi.FsmInstr, abi.Proposal, abi.LeaderEntry,
                                  abi.StepArgs, abi.ReplicaState)]
    assert got == want
    for name, size in abi.EXPECTED_SIZES.items():
        assert C.sizeof(getattr(abi, name)) == size


def test_election_timeout_is_the_same_function_everywhere(engine_lib, oracle_lib):
    """Deviation D2 is normative: the engine library (host symbol), the oracle and the
    ABI text must agree."""
    engine_lib.jr_election_timeout.argtypes = [C.c_uint64, C.c_uint64] + [C.c_uint32] * 4
    engine_lib.jr_election_timeout.restype = C.c_uint32
    for seed, g, n, d in [(0, 0, 1, 0), (1, 65535, 5, 3), (2**63, 2**40, 7, 1000)]:
        assert engine_lib.jr_election_timeout(seed, g, n, d, 500, 1000) == \
            oracle_lib.jro_election_timeout(seed, g, n, d, 500, 1000)


def test_engine_library_is_sm100a_cuda(engine_lib):
    # the toolkit build() compiled with, when it is not on PATH
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", ENGINE_LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def test_create_without_gpu_fails_loudly(engine_lib):
    """No CPU fallback: on a box without a CUDA device creation must fail, not emulate."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cfg = abi.default_config(4, 3)
    h = C.c_void_p()
    engine_lib.jr_engine_create.restype = C.c_int
    st = engine_lib.jr_engine_create(C.byref(cfg), C.byref(h))
    assert st in (abi.E_NO_DEVICE, abi.E_CUDA)
    assert not h.value


def test_package_refuses_the_emulation_library():
    """The CPU emulation of the device code (tests/emu) is test infrastructure; pointing the
    package at it must fail loudly rather than become a CPU fallback."""
    from josefine_b200.raft import RaftError, _open_engine_library
    from tests.emu import emu
    emu.load()
    with pytest.raises(RaftError) as e:
        _open_engine_library(emu.LIB_PATH)
    assert "no CPU fallback" in str(e.value)
