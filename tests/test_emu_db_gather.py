"""Reading a resident database's subjects back by caller id (psb_db_align, psb_db_subject): pack_db_kernel packs
random subjects at 2, 3 and 5 bit in a random storage order, invert_perm_kernel inverts that order and
unpack_db_kernel gathers caller-order ids through it; the result must be the mapped residues byte for byte.
The kernel sources run on the CPU under -DPSB_EMULATE (tests/emu/db_gather_check.cpp); no GPU."""
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("dbg") / "db_gather_check")
    subprocess.run(["g++", "-O1", "-std=c++20", "-pthread", "-o", exe, os.path.join(HERE, "emu", "db_gather_check.cpp")], check=True)
    return exe


@pytest.mark.parametrize("bits", [2, 3, 5])
@pytest.mark.parametrize("seed,n", [(1, 1), (2, 7), (3, 257)])
def test_gather_by_caller_id(checker, bits, seed, n):
    r = subprocess.run([checker, str(seed), str(bits), str(n)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("ok"), r.stdout + r.stderr
