"""The substream coder of blocked containers (cbc_b200/csrc/k2_roles.cuh) is plain scalar host + device code: the
same source the GPU threads run is compiled for the CPU here (tests/native/test_k2_roles.cpp) and must write the
oracle's container byte for byte -- cold blocks, generation-primed blocks (with a host restatement of the merge kernels
over the same memory layouts), fixed and variable length, several chromosomes, sparse coverage (every POS an escape) --
and decode it back to the input's edit records. The oracle is the checker here; the product never links it."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_build", "test_k2_roles")


@pytest.fixture(scope="module")
def harness():
    os.makedirs(os.path.dirname(BIN), exist_ok=True)
    cmd = ["g++", "-O1", "-std=c++17", "-Wall", "-Wno-unused-function", "-Iinclude", "-Icbc_b200/csrc", "-Icbc_b200/csrc/host", "-Ioracle",
           "tests/native/test_k2_roles.cpp", "cbc_b200/csrc/host/synth.c", "oracle/cbc_oracle.c", "-o", BIN]
    subprocess.run(cmd, cwd=ROOT, check=True)
    return BIN


CASES = [
    # seed n_reads genome len_min len_max p_sub p_indel p_clip gen_mode [block_reads [n_chr [n_flags [random_head]]]]
    "5 20000 300000 150 150 0.005 0 0 0 512",
    "6 20000 300000 150 150 0.005 0 0 1",
    "7 30000 400000 100 100 0.01 0.002 0.05 0 777",
    "8 30000 400000 100 100 0.01 0.002 0.05 1",
    "9 40000 500000 50 250 0.005 0.02 0.3 1",
    "10 40000 500000 50 250 0.005 0.02 0.3 0 300",
    "11 30000 600000 100 100 0.01 0.001 0 1 4294967295 3",
    "12 5000 40000000 100 100 0.01 0 0 1",
    "13 5000 40000000 100 100 0.01 0 0 0 200",
    "14 400000 2000000 150 150 0.005 0.001 0.01 1",
    "15 400000 2000000 100 100 0.02 0 0 0 100000",
    "16 1 100000 100 100 0.01 0 0 1",
    "17 3 100000 100 100 0.01 0 0 0 2",
    # more distinct FLAG values than a block adapts / a snapshot keeps (rules F1 / F2, cbcg_format.h)
    "18 30000 300000 100 100 0.01 0 0 0 4000 1 300",
    "19 30000 300000 100 100 0.01 0 0 1 4294967295 1 300",
    "20 60000 400000 100 100 0.01 0.001 0 1 4294967295 1 1500",
    "21 20000 300000 100 100 0.01 0 0 0 20000 1 3000",
    "22 60000 400000 100 100 0.01 0 0 1 4294967295 1 1500 1",   # the blocks of a generation adapt different values: the merge keeps 256 (F2)
    "23 200000 1000000 100 100 0.01 0 0 1 4294967295 1 400 1",
    # 12 reads over 60 Mb in one block: POS steps of several Mb, above the single stream's 5 M limit
    "24 12 60000000 100 100 0.01 0 0 0 12",
    "25 12 60000000 100 100 0.01 0 0 1",
]


@pytest.mark.parametrize("case", CASES)
def test_roles_write_and_read_the_oracles_container(harness, case):
    p = subprocess.run([harness] + case.split(), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    assert p.stdout.startswith("ok:")
