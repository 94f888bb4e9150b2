"""SURVEY.md 8f-2, first slice: the joint-limit half of Constraints::linearizeConstraints on the device
(rbt_linearize_joint_limits: PDIPM residuals of the box rows + their dual terms in the gradients).
CPU: the oracle against what the reference's own JointPosition / Velocity / Torques Lower / Upper Limit classes (compiled
unmodified, oracle/Makefile.ref) computed on the same problems (tests/golden/golden_ref_stage_r2.npz, "jl_" keys, made by
make_golden_ref_stage.py), and against a numpy statement of their formulas;
GPU: the CUDA kernel against the oracle."""
import ctypes
import os
import sys

import numpy as np
import pytest

import oracle_lib
from helpers import small_event_schedule, trot_schedule
from robotoc_b200 import ANYMAL, StageLayout
from robotoc_b200.grid import IMPACT, TERMINAL

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import golden_io  # noqa: E402
from make_golden_ref_stage import JOINT_LIMIT_PROBLEMS, joint_limit_problem  # noqa: E402


def _oracle(lib, table, sd, ctrl, bound, sol, lin, con):
    l, c = lin.copy(), con.copy()
    csd = sd.c()
    P = oracle_lib.ptr
    lib.orc_linearize_joint_limits_batch(ctypes.byref(csd), ctypes.byref(table), ctrl, len(ctrl), lin.shape[0], P(bound), P(sol), P(l), P(c))
    return l, c


def _numpy(table, S, ctrl, bound, sol, lin, con):
    """joint_*_limit.cpp:47-63: residual = sign (x - bound) + slack; l_x += sign dual; levels gated by the grid index."""
    l, c = lin.copy(), con.copy()
    nv = S.nv
    for i, ct in enumerate(ctrl):
        if ct.type in (IMPACT, TERMINAL):
            continue
        for r in range(table.n_box):
            br = table.box[r]
            if {0: 2, 1: 1}.get(br.var, 0) + ct.ineq_gate > 2:
                continue
            x = {0: sol[:, i, S.s_q + br.idx + 1], 1: sol[:, i, S.s_v + br.idx], 2: sol[:, i, S.s_a + br.idx], 3: sol[:, i, S.s_u + br.idx]}[br.var]
            g = {0: S.l_lx + br.idx, 1: S.l_lx + nv + br.idx, 2: S.l_la + br.idx, 3: S.l_lu + br.idx}[br.var]
            c[:, i, S.c_res + r] = br.sign * (x - bound[r]) + con[:, i, S.c_slack + r]
            l[:, i, g] += br.sign * con[:, i, S.c_dual + r]
    return l, c


@pytest.mark.parametrize("which", list(JOINT_LIMIT_PROBLEMS))
def test_oracle_joint_limit_linearisation(which):
    sched, batch, seed = JOINT_LIMIT_PROBLEMS[which]
    lib, table, sd, S, ctrl, lin, con, sol, bound = joint_limit_problem(sched(), batch, seed)
    l_o, c_o = _oracle(lib, table, sd, ctrl, bound, sol, lin, con)
    l_n, c_n = _numpy(table, S, ctrl, bound, sol, lin, con)
    np.testing.assert_allclose(l_o, l_n, rtol=1e-15, atol=1e-15)
    np.testing.assert_allclose(c_o, c_n, rtol=1e-15, atol=1e-15)
    assert np.abs(l_o - lin).max() > 0.01 and np.abs(c_o - con).max() > 0.1   # it did something
    assert np.array_equal(c_o[:, 0, S.c_res:S.c_res + 48], con[:, 0, S.c_res:S.c_res + 48])  # stage 0: position / velocity rows gated
    # the reference's classes, stored as what they changed: every entry they left alone, a sample of the ones they set
    G = golden_io.load(os.path.join(HERE, "golden", "golden_ref_stage_r2.npz"))
    for got, inp, delta in ((l_o, lin, G[f"jl_{which}_dlin"]), (c_o, con, G[f"jl_{which}_dcon"])):
        m = golden_io.finite(delta)
        assert m.any() and np.any(delta[m] != 0.0)
        np.testing.assert_allclose(got[m], (inp + delta)[m], rtol=1e-14, atol=1e-14)


@pytest.mark.gpu
@pytest.mark.parametrize("which,batch", [("small_sto", 3), ("trot", 16)])
def test_cuda_joint_limit_linearisation_matches_the_oracle(which, batch):
    from robotoc_b200 import DirectMultipleShooting, RiccatiRecursion
    sched = {"small_sto": small_event_schedule(True), "trot": trot_schedule(40)}[which]
    lib, table, sd, S, ctrl, lin, con, sol, bound = joint_limit_problem(sched, batch, 82)
    S = StageLayout(sd)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), batch)
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    with pytest.raises(RuntimeError):
        dms.linearizeJointLimits()  # limits not set yet
    dms.setJointLimits(bound)
    dms._up(6, lin, S.l_stride, None)
    dms.setConstraintData(con)
    dms.setSolution(sol)
    dms.linearizeJointLimits()
    l_o, c_o = _oracle(lib, table, sd, ctrl, bound, sol, lin, con)
    np.testing.assert_array_equal(dms._down(6, lin.shape), l_o)
    np.testing.assert_array_equal(dms.getConstraintData(), c_o)
    rr.close()
