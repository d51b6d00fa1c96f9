"""The plan bytes committed for traced OperateOn closures (tests/golden/plans/make_fn_plans.py, compared byte for byte
by julia/test_plans.jl) must be what host/lowering.py emits today, parse as the layout of include/signalops.h, and
hold the closure-function opcodes they were made to pin."""
import os
import struct
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden", "plans"))
import make_fn_plans  # noqa: E402


@pytest.mark.parametrize("name", sorted(make_fn_plans.CASES))
def test_committed_fn_plan_bytes_are_current(name):
    with open(os.path.join(HERE, "golden", "plans", name + ".bin"), "rb") as f:
        want = f.read()
    assert make_fn_plans.plan_bytes(name) == want, (
        f"{name}: lowering.py no longer emits the committed plan; rerun tests/golden/plans/make_fn_plans.py "
        "and update julia/test_plans.jl if the format changed")


@pytest.mark.parametrize("name", sorted(make_fn_plans.CASES))
def test_fn_plan_sections_add_up(name):
    b = make_fn_plans.plan_bytes(name)
    magic, ver, n_in, n_tmp, n_out, n_scal, n_tab, n_instr, n_piece, n_stage, n_dbl = struct.unpack_from("<10IQ", b, 0)
    assert magic == 0x504F4753 and ver == 1
    assert len(b) == 48 + 16 * (n_in + n_tmp + n_out) + 16 * n_tab + 80 * n_instr + 32 * n_piece + 128 * n_stage + 8 * n_dbl
    o = 48 + 16 * (n_in + n_tmp + n_out) + 16 * n_tab
    ops = [b[o + 80 * k] for k in range(n_instr)]
    # every case but mid/side (plain arithmetic of a whole-frame closure) applies a closure function
    assert (name == "midside") != any(op in (14, 15, 16) for op in ops)
