"""SURVEY.md 8f-3: batched trial step sizes + the filter acceptance loop of robotoc::LineSearch.
CPU: the oracle's filter loop against what the reference's own LineSearchFilter class (compiled unmodified, oracle/Makefile.ref)
     accepted over many consecutive line searches (tests/golden/golden_ref_seeds.npz, made by make_golden_ref.py); the
     oracle's trial solutions against its own update at the same step size.
GPU: the CUDA path against the oracle."""
import ctypes
import os
import sys

import numpy as np
import pytest

import oracle_lib
from helpers import small_event_schedule, trot_schedule
from iteration_check import oracle_iteration
from robotoc_b200 import ANYMAL, Layout, StageDims, StageLayout, anymal_constraint_table
from robotoc_b200.grid import IMPACT, TERMINAL
from synth import make_stage_inputs

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import golden_io  # noqa: E402
import make_golden_ref as mg  # noqa: E402

T_Q, T_V, T_A, T_U, T_F, T_STRIDE = 0, 20, 38, 56, 68, 80
CAP = 16


def _orc():
    lib = oracle_lib.load()
    vp, ci, cd = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    lib.orc_trial_batch.argtypes = [vp, vp, vp, ci, ci, ci, cd] + [vp] * 8
    lib.orc_line_search_filter.argtypes = [ci, ci, cd, cd, cd, cd, ci] + [vp] * 10
    return lib


def _filter_oracle(lib, steps, cost0, viol0, cost, barrier, viol, filt, nfilt, rate=0.75, min_step=0.05, cr=0.005, vr=0.005):
    n_trials, batch = cost.shape
    out_step, out_k = np.zeros(batch), np.zeros(batch, dtype=np.int32)
    P = oracle_lib.ptr
    lib.orc_line_search_filter(batch, n_trials, rate, min_step, cr, vr, CAP, P(steps), P(cost0), P(viol0), P(cost), P(barrier), P(viol),
                               P(filt), nfilt.ctypes.data_as(ctypes.c_void_p), P(out_step), out_k.ctypes.data_as(ctypes.c_void_p))
    return out_step, out_k


def test_oracle_filter_loop_equals_the_reference_line_search_filter():
    lib = _orc()
    G = golden_io.load(os.path.join(HERE, "golden", "golden_ref_seeds.npz"))
    f = mg.FILTER
    for case, (amax, cost0, viol0, cost, viol) in enumerate(mg.filter_cases()):
        step_r, k_r = G["filter_step"][case], G["filter_k"][case]
        # the oracle: one "OCP" (batch 1) whose filter persists across the rounds
        filt, nfilt = np.zeros((1, 2 * CAP)), np.zeros(1, dtype=np.int32)
        for r in range(f["rounds"]):
            steps = np.array([[amax[r], 1.0]])
            st, kk = _filter_oracle(lib, steps, cost0[r:r + 1].copy(), viol0[r:r + 1].copy(), np.ascontiguousarray(cost[r][:, None]),
                                    np.zeros((f["n_trials"], 1)), np.ascontiguousarray(viol[r][:, None]), filt, nfilt, rate=f["rate"],
                                    min_step=f["min_step"], cr=f["cost_reduction"], vr=f["violation_reduction"])
            assert kk[0] == k_r[r] and st[0] == step_r[r], (case, r)
        assert nfilt[0] <= CAP


def _problem(sched, batch, seed, getter=True, impact_cones=False):
    lib = _orc()
    table = anymal_constraint_table(impact_friction_cone=impact_cones)
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S = StageLayout(sd, getter=lib.orc_stage_layout_get)
    K = Layout(ANYMAL, getter=lib.orc_layout_get)
    td, ev, ctrl = sched
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, batch, seed, impact_cones=impact_cones)
    ref = oracle_iteration(sd, S, K, table, ctrl, lin, con, sol, dx0)
    return lib, table, sd, S, K, ctrl, lin, con, sol, dx0, ref


def _oracle_trials(lib, sd, table, ctrl, S, K, sol, ref, n_trials, rate=0.75):
    batch, n_grid = sol.shape[0], sol.shape[1]
    alphas, barrier = np.zeros((n_trials, batch)), np.zeros((n_trials, batch))
    trial = np.zeros((n_trials, batch, n_grid, T_STRIDE))
    csd = sd.c()
    P = oracle_lib.ptr
    lib.orc_trial_batch(ctypes.byref(csd), ctypes.byref(table), ctrl, n_grid, batch, n_trials, rate, P(sol), P(ref["d"]), P(ref["xd_exp"]),
                        P(ref["cc_exp"]), P(ref["steps"]), P(alphas), P(trial), P(barrier))
    return alphas, barrier, trial


@pytest.mark.parametrize("impact_cones", [False, True])
def test_oracle_trial_zero_is_the_primal_part_of_the_update(impact_cones):
    """Trial k = 0 uses alpha_max, the step the update takes: its q, v, a | dv, u, f are the updated solution's."""
    lib, table, sd, S, K, ctrl, lin, con, sol, dx0, ref = _problem(small_event_schedule(True), 2, 71, impact_cones=impact_cones)
    alphas, barrier, trial = _oracle_trials(lib, sd, table, ctrl, S, K, sol, ref, 3)
    np.testing.assert_array_equal(alphas[0], ref["steps"][:, 0])
    np.testing.assert_allclose(alphas[2], ref["steps"][:, 0] * 0.75 ** 2, rtol=1e-15)
    for i, c in enumerate(ctrl):
        new = ref["sol"][:, i]
        np.testing.assert_allclose(trial[0, :, i, T_Q:T_Q + S.nq], new[:, S.s_q:S.s_q + S.nq], rtol=0, atol=1e-14)
        np.testing.assert_allclose(trial[0, :, i, T_V:T_V + 18], new[:, S.s_v:S.s_v + 18], rtol=0, atol=1e-14)
        if c.type == TERMINAL:
            continue
        a_new = new[:, S.s_dv:S.s_dv + 18] if c.type == IMPACT else new[:, S.s_a:S.s_a + 18]
        np.testing.assert_allclose(trial[0, :, i, T_A:T_A + 18], a_new, rtol=0, atol=1e-14)
        np.testing.assert_allclose(trial[0, :, i, T_F:T_F + c.nf], new[:, S.s_f:S.s_f + c.nf], rtol=0, atol=1e-14)
        if c.type != IMPACT:
            np.testing.assert_allclose(trial[0, :, i, T_U:T_U + 12], new[:, S.s_u:S.s_u + 12], rtol=0, atol=1e-14)
    # barrier of trial 0 == log barrier of the updated slacks
    lb = np.zeros(2)
    for i, c in enumerate(ctrl):
        if c.type == TERMINAL or (c.type == IMPACT and not impact_cones):
            continue
        act = np.ones(S.nc, dtype=bool)
        if c.type == IMPACT:
            act[:S.nbox] = False
        for r in range(S.nbox):
            if {0: 2, 1: 1}.get(table.box[r].var, 0) + c.ineq_gate > 2:
                act[r] = False
        for ci in range(S.ncon):
            if not (c.contact_mask >> ci) & 1:
                act[S.nbox + 5 * ci:S.nbox + 5 * ci + 5] = False
        lb += -table.barrier * np.sum(np.log(ref["cc_upd"][:, i, S.c_slack:S.c_slack + S.nc][:, act]), axis=1)
    np.testing.assert_allclose(barrier[0], lb, rtol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("which,batch", [("small_sto", 3), ("trot", 8), ("trot_icone", 4)])
def test_cuda_line_search_matches_the_oracle(which, batch):
    from robotoc_b200 import DirectMultipleShooting, LineSearch, RiccatiRecursion
    sched = {"small_sto": small_event_schedule(True), "trot": trot_schedule(40), "trot_icone": trot_schedule(40)}[which]
    lib, table, sd, S, K, ctrl, lin, con, sol, dx0, ref = _problem(sched, batch, 72, impact_cones=which.endswith("icone"))
    S = StageLayout(sd)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), batch)
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    dms.condense(lin, con)
    rr.backwardRiccatiRecursion()
    rr.forwardRiccatiRecursion(dx0)
    dms.computeStepSizes()
    dms._up(9, sol, S.s_stride, None)  # the current iterate (trials are generated BEFORE integrateSolution)
    ls = LineSearch(dms)
    n_trials = 6
    alphas, barrier, trial = ls.trialSolutions(n_trials)
    a_o, b_o, t_o = _oracle_trials(lib, sd, table, ctrl, S, K, sol, ref, n_trials)
    np.testing.assert_allclose(alphas, a_o, rtol=1e-14)
    np.testing.assert_allclose(barrier, b_o, rtol=1e-11)
    np.testing.assert_allclose(trial, t_o, rtol=0, atol=1e-11 * max(1.0, np.abs(t_o).max()))
    # the acceptance loop, several consecutive line searches with persistent per-OCP filters
    rng = np.random.default_rng(9)
    filt, nfilt = np.zeros((batch, 2 * CAP)), np.zeros(batch, dtype=np.int32)
    ls.clearHistory()
    steps = np.ascontiguousarray(ref["steps"])
    for rnd in range(6):
        nt = ls.numTrials(dms.maxPrimalStepSize())
        al, bar, _ = ls.trialSolutions(nt, want_trials=False)
        cost = np.ascontiguousarray(5.0 - rnd + rng.normal(0, 0.5, size=(nt, batch)))
        viol = np.ascontiguousarray(np.abs(0.5 - 0.05 * rnd + rng.normal(0, 0.05, size=(nt, batch))))
        cost0, viol0 = cost[0] + 0.1, viol[0] + 0.01
        got_step, got_k = ls.computeStepSize(cost0, viol0, lambda tr, a: (cost, viol))
        want_step, want_k = _filter_oracle(lib, steps, cost0.copy(), viol0.copy(), cost, np.ascontiguousarray(bar), viol, filt, nfilt)
        np.testing.assert_array_equal(got_k, want_k)
        np.testing.assert_allclose(got_step, want_step, rtol=1e-12)  # alpha_max comes from the device / the oracle: equal to rounding
    rr.close()
