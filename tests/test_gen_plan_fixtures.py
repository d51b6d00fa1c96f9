"""The plan bytes committed for traced generator closures (tests/golden/plans/make_gen_plans.py, compared byte for byte
by julia/test_gen_plans.jl) must be what host/lowering.py emits today, and hold device generators only: no input
buffer carries a generator's frames."""
import os
import struct
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden", "plans"))
import make_gen_plans  # noqa: E402


@pytest.mark.parametrize("name", sorted(make_gen_plans.CASES))
def test_committed_gen_plan_bytes_are_current(name):
    with open(os.path.join(HERE, "golden", "plans", name + ".bin"), "rb") as f:
        want = f.read()
    assert make_gen_plans.plan_bytes(name) == want, (
        f"{name}: lowering.py no longer emits the committed plan; rerun tests/golden/plans/make_gen_plans.py "
        "and check julia/test_gen_plans.jl")


@pytest.mark.parametrize("name", sorted(make_gen_plans.CASES))
def test_gen_plan_reads_no_generator_frames(name):
    b = make_gen_plans.plan_bytes(name)
    magic, ver, n_in, n_tmp, n_out, n_scal, n_tab, n_instr, n_piece, n_stage, n_dbl = struct.unpack_from("<10IQ", b, 0)
    assert magic == 0x504F4753 and ver == 1
    assert len(b) == 48 + 16 * (n_in + n_tmp + n_out) + 16 * n_tab + 80 * n_instr + 32 * n_piece + 128 * n_stage + 8 * n_dbl
    assert n_in == (1 if name == "gen_am" else 0)          # gen_am's one input is its noise
    o = 48 + 16 * (n_in + n_tmp + n_out) + 16 * n_tab
    leaves = [b[o + 80 * k + 1] for k in range(n_instr)]
    assert 4 in leaves                                      # SIGOPS_LEAF_GEN
