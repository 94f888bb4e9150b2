"""Odd contact dimensions and the general-Fxx backward sweep.

The ANYmal crawl (helpers.crawl_schedule, examples/anymal/crawl.cpp) is the schedule with three feet in contact (nf = 9, an odd
[a; f] height nv + nf = 27), single-foot impacts (nf = 3 on the Impact stage, nv + nf = 21) and switching constraints with
ns = 3 -- extents the other schedules (nf, ns in {0, 6, 12}) never reach:
  CPU: the oracle's Riccati direction on crawl_small solves the dense block KKT system; the oracle == the reference's code on
       the crawl schedules runs through the FIELD_CASES / SEED_CASES of test_golden_ref.py / test_golden_ref_stage.py;
  GPU: the Riccati API, the stage layer (with NaN in the inactive rows of J), rbt_eval_kkt and the line-search trials == the
       oracle, the CUDA path == the reference's fixtures, and a 131-OCP batch (4 host chunks).
The Riccati-only API picks the backward instance that skips the structural rows of Fxx (RBT_FXX_MECHANICAL) or the general
one; under RBT_FXX_AUTO a device check decides.  GPU: records that are not mechanical -- everywhere, or in one entry -- must
give the general instance's (the oracle's) answer."""
import ctypes

import numpy as np
import pytest

import oracle_lib
from helpers import crawl_schedule, dense_kkt_solve, rel_err, small_event_schedule, trot_schedule
from robotoc_b200 import ANYMAL, Layout
from robotoc_b200.grid import IMPACT, LIFT, TERMINAL
from synth import make_kkt

TOL = 1e-8
FXX_AUTO, FXX_MECHANICAL, FXX_GENERAL = 0, 1, 2   # include/robotoc_b200.h


# ---- CPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size,n_grid", [("crawl_small", 31), ("crawl_full", 219)])
@pytest.mark.parametrize("sto", [False, True])
def test_crawl_schedule_has_the_odd_contact_dimensions(size, n_grid, sto):
    td, ev, ctrl = crawl_schedule(size, sto=sto)
    cycles = {"crawl_small": 1, "crawl_full": 2}[size]
    assert len(ctrl) == n_grid and td.N == {"crawl_small": 26, "crawl_full": 210}[size]
    impacts = [i for i, c in enumerate(ctrl) if c.type == IMPACT]
    assert len(impacts) == 4 * cycles and sum(c.type == LIFT for c in ctrl) == 2 * cycles
    for i in impacts:
        assert ctrl[i].nf == 3 and ctrl[i].ns == 0 and bin(ctrl[i].contact_mask).count("1") == 1
        assert ctrl[i - 2].ns == 3 and ctrl[i - 2].type not in (IMPACT, LIFT)  # the switching constraint of the impact
    assert sorted(i for i, c in enumerate(ctrl) if c.ns > 0) == [i - 2 for i in impacts]
    assert {c.nf for c in ctrl if c.type != IMPACT and c.type != TERMINAL} == {9, 12}
    assert all(c.nf == 9 for c in ctrl if c.type == LIFT)
    assert {c.contact_mask for c in ctrl if c.nf == 9} == {0b0111, 0b1011, 0b1101, 0b1110}
    assert all(bool(c.sto) == sto for c in ctrl[:-2])


@pytest.mark.parametrize("seed", [35, 36])
def test_oracle_direction_solves_the_dense_kkt_system_of_the_crawl(seed):
    """crawl_small as one dense block KKT system (helpers.dense_kkt_solve): the oracle's Riccati direction solves it, incl.
    the multipliers xi of the ns = 3 switching constraints."""
    L = Layout(ANYMAL)
    td, ev, ctrl = crawl_schedule("crawl_small")
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=2, seed=seed)
    kk, ric, d, info = oracle_lib.riccati_batch(ANYMAL, L, ctrl, kkt, dx0)
    assert info == 0
    n_xi = 0
    for b in range(2):
        ref = dense_kkt_solve(ANYMAL, L, ctrl, kkt[b], dx0[b])
        for i, c in enumerate(ctrl):
            di = d[b, i]
            assert rel_err(di[L.d_dx:L.d_dx + ANYMAL.nx], ref[("dx", i)]) < 1e-9, ("dx", i)
            assert rel_err(di[L.d_dlmdgmm:L.d_dlmdgmm + ANYMAL.nx], ref[("lmd", i)]) < 1e-9, ("lmd", i)
            if ("du", i) in ref:
                assert rel_err(di[L.d_du:L.d_du + ANYMAL.nu], ref[("du", i)]) < 1e-9, ("du", i)
            if ("xi", i) in ref:
                assert c.ns == 3
                assert rel_err(di[L.d_dxi:L.d_dxi + c.ns], ref[("xi", i)]) < 1e-9, ("xi", i)
                n_xi += 1
    assert n_xi == 2 * 4


# ---- GPU: the crawl through every layer ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("size,sto,seed", [("crawl_small", False, 41), ("crawl_small", True, 42), ("crawl_full", False, 43)])
def test_cuda_riccati_api_on_the_crawl(size, sto, seed):
    """P, s, K, k, M, m, the STO terms, F, H, G, lu and the direction (dxi at ns = 3) of every stage == the oracle."""
    from test_gpu_parity import _run_case
    td, ev, ctrl = crawl_schedule(size, sto=sto)
    _run_case(ctrl, batch=3, seed=seed)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["crawl_small", "crawl_small_sto"])
def test_cuda_riccati_api_reproduces_the_reference_crawl_fixture(name):
    import test_golden_ref as tg
    from robotoc_b200 import RiccatiRecursion
    L = Layout(ANYMAL)
    ctrl, kkt, dx0 = tg.mg.field_inputs(name, tg.mg.FIELD_CASES[name], L)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), kkt.shape[0])
    rr.setTimeDiscretization(ctrl)
    rr.backwardRiccatiRecursion(kkt)
    rr.forwardRiccatiRecursion(dx0)
    assert int(rr.info().max()) == 0
    kk_r, ric_r, d_r = tg.field_fixture(name)
    tg.assert_every_field(L, ctrl, None, rr.getRiccatiFactorization(), rr.getDirection(), kk_r, ric_r, d_r, tol=TOL)
    rr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("size,sto,icone,batch,seed", [("crawl_small", False, False, 3, 51), ("crawl_small", False, True, 3, 52),
                                                       ("crawl_small", True, False, 3, 53), ("crawl_full", False, False, 2, 54)])
def test_cuda_stage_layer_on_the_crawl(size, sto, icone, batch, seed):
    """condense, backward / forward, expand_and_step_sizes, update: every record after every call == the oracle (daf and
    dbetamu over their nv + nf rows); the one-call host paths (dense 1 / 3 chunks, wire, wire with RBT_COST_ROBOTOC,
    resident) give the same bits.  The device's records carry NaN in the inactive rows of J (nf = 9 and 3 leave 3 and 9)."""
    from test_gpu_stage import _run
    td, ev, ctrl = crawl_schedule(size, sto=sto)
    _run(ctrl, batch=batch, seed=seed, impact_cones=icone, poison=True)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["crawl_small", "crawl_small_sto", "crawl_small_icone"])
def test_cuda_stage_layer_reproduces_the_reference_crawl_fixture(which):
    import test_golden_ref_stage as tg
    from robotoc_b200 import DirectMultipleShooting, RiccatiRecursion
    from iteration_check import reference_view_of_expansion
    from test_gpu_stage import poison_inactive_contact_rows
    table, sd, S, K, ctrl, lin, con, sol, dx0 = tg.mg.seed_problem(which, tg.mg.SEED_CASES[which])
    rr = RiccatiRecursion(ANYMAL, len(ctrl), lin.shape[0])
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    dms.condense(poison_inactive_contact_rows(S, ctrl, lin), con)
    got = dict(kkt=dms.getKKT(), cc_cond=dms.getConstraintData())
    rr.backwardRiccatiRecursion()
    rr.forwardRiccatiRecursion(dx0)
    assert int(rr.info().max()) == 0
    got["ric"] = rr.getRiccatiFactorization()
    dms.computeStepSizes()
    got["steps"] = np.stack([dms.maxPrimalStepSize(), dms.maxDualStepSize()], axis=1)
    got["cc_exp"], got["xd_exp"] = dms.getConstraintData(), dms.getExpandedDirection()
    dms.integrateSolution(sol)
    got["d_upd"], got["xd_upd"], got["cc_upd"], got["ex_upd"] = (rr.getDirection(), dms.getExpandedDirection(), dms.getConstraintData(),
                                                                 reference_view_of_expansion(S, dms.getExpansionData()))
    ref = tg.golden_io.load(tg.mg.seed_path(which))
    tg._cmp_records(S, K, ctrl, got, ref, TOL, impact_cones=which.endswith("_icone"))
    rr.close()


@pytest.mark.gpu
def test_cuda_stage_layer_crawl_batch_131_every_ocp():
    """131 OCPs (a prime above the 128 at which the one-call host path splits the batch into 4 chunks): the full iteration on
    every OCP (condition-aware, iteration_check.py), and the chunked one-call path gives the same bits."""
    from iteration_check import compare_final, oracle_iteration, oracle_sensitivity, run_device_iteration
    from robotoc_b200 import DirectMultipleShooting, RiccatiRecursion, StageDims, StageLayout, anymal_constraint_table
    from synth import make_stage_inputs
    td, ev, ctrl = crawl_schedule("crawl_small")
    table = anymal_constraint_table()
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S, K = StageLayout(sd), Layout(ANYMAL)
    batch = 131
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, batch, 55)
    ref = oracle_iteration(sd, S, K, table, ctrl, lin, con, sol, dx0)
    sens = oracle_sensitivity(sd, S, K, table, ctrl, lin, con, sol, dx0, ref)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), batch)
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    got = run_device_iteration(rr, dms, lin, con, sol, dx0)
    assert int(got["info"].max()) == 0
    compare_final(S, K, ctrl, ref, got["ric"], got["d"], got["steps"], got["sol"], got["cc"], TOL, sensitivity=sens)
    sol2, con2, steps2 = dms.iteration_host(lin, con, sol, dx0)
    used = S.s_xi + S.nsm
    np.testing.assert_array_equal(sol2[:, :, :used], got["sol"][:, :, :used])
    np.testing.assert_array_equal(steps2, got["steps"])
    rr.close()


@pytest.mark.gpu
def test_cuda_eval_kkt_on_the_crawl():
    from robotoc_b200 import DirectMultipleShooting, RiccatiRecursion, StageLayout
    from test_eval_rows import _oracle_perf, _setup
    batch = 3
    lib, table, sd, S, ctrl, lin, con, sol, dx0 = _setup(crawl_schedule("crawl_small"), batch, 61)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), batch)
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    got = dms.evalKKT(lin, con)
    want = _oracle_perf(lib, sd, table, ctrl, lin, con)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    assert (want[:, 3] > 0).all()  # the ns = 3 switching residuals are part of the primal feasibility
    rr.close()


@pytest.mark.gpu
def test_cuda_line_search_trials_on_the_crawl():
    from robotoc_b200 import DirectMultipleShooting, LineSearch, RiccatiRecursion, StageLayout
    from test_line_search import _oracle_trials, _problem
    batch = 3
    lib, table, sd, S, K, ctrl, lin, con, sol, dx0, ref = _problem(crawl_schedule("crawl_small"), batch, 62)
    S = StageLayout(sd)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), batch)
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    dms.condense(lin, con)
    rr.backwardRiccatiRecursion()
    rr.forwardRiccatiRecursion(dx0)
    dms.computeStepSizes()
    dms._up(9, sol, S.s_stride, None)  # the current iterate (trials are generated before integrateSolution)
    n_trials = 6
    alphas, barrier, trial = LineSearch(dms).trialSolutions(n_trials)
    a_o, b_o, t_o = _oracle_trials(lib, sd, table, ctrl, S, K, sol, ref, n_trials)
    np.testing.assert_allclose(alphas, a_o, rtol=1e-14)
    np.testing.assert_allclose(barrier, b_o, rtol=1e-11)
    np.testing.assert_allclose(trial, t_o, rtol=0, atol=1e-11 * max(1.0, np.abs(t_o).max()))
    rr.close()


# ---- GPU: the general-Fxx backward instance and its dispatch --------------------------------------------------------------
def _fxx(L, kkt, i, r, c):
    """View index of Fxx[r, c] of grid point i (column-major nx x nx)."""
    return (slice(None), i, L.k_Fxx + r + c * ANYMAL.nx)


def _non_mechanical(L, ctrl, kkt, seed):
    """kkt + 1e-2 U(-1,1) on the rows nv_passive..nv-1 of Fqq and Fqv of every non-terminal grid point: the rows the mechanical
    instance takes as [e_r^T, dt e_r^T] without reading them."""
    out = kkt.copy()
    rng = np.random.default_rng(seed)
    nv, nx = ANYMAL.nv, ANYMAL.nx
    for i, c in enumerate(ctrl):
        if c.type == TERMINAL:
            continue
        F = out[:, i, L.k_Fxx:L.k_Fxx + nx * nx].reshape(-1, nx, nx)  # [batch, col, row]
        F[:, :, 6:nv] += 1e-2 * rng.uniform(-1.0, 1.0, size=(out.shape[0], nx, nv - 6))
    return out


def _solve(ctrl, kkt, dx0, mode):
    from robotoc_b200 import RiccatiRecursion
    rr = RiccatiRecursion(ANYMAL, len(ctrl), kkt.shape[0])
    rr.setTimeDiscretization(ctrl)
    if mode is not None:
        assert rr._lib.rbt_set_fxx_structure(rr._h, mode) == 0
    rr.backwardRiccatiRecursion(kkt, write_fact=True)
    rr.forwardRiccatiRecursion(dx0)
    out = rr.getRiccatiFactorization(), rr.getDirection(), rr.getFactorizedKKT()
    assert int(rr.info().max()) == 0
    rr.close()
    return out


def _oracle(L, ctrl, kkt, dx0):
    kk, ric, d, info = oracle_lib.riccati_batch(ANYMAL, L, ctrl, kkt, dx0)
    assert info == 0
    return kk, ric, d


def _assert_oracle(L, ctrl, got, ref):
    from test_gpu_parity import _compare
    _compare(ANYMAL, L, ctrl, got[0], ref[1], got[1], ref[2], got[2], ref[0], tol=TOL)


def _deviation(L, ctrl, got, ref):
    """Largest stage-wise relative difference of P and dx."""
    nx = ANYMAL.nx
    return max(max(rel_err(got[0][:, i, L.r_P:L.r_P + nx * nx], ref[1][:, i, L.r_P:L.r_P + nx * nx]),
                   rel_err(got[1][:, i, L.d_dx:L.d_dx + nx], ref[2][:, i, L.d_dx:L.d_dx + nx])) for i in range(len(ctrl)))


FXX_SCHEDULES = {"small": lambda: small_event_schedule(False), "small_sto": lambda: small_event_schedule(True),
                 "trot_n40": lambda: trot_schedule(40), "crawl_small_sto": lambda: crawl_schedule("crawl_small", sto=True)}


@pytest.mark.gpu
@pytest.mark.parametrize("which", list(FXX_SCHEDULES))
@pytest.mark.parametrize("batch", [1, 37])
def test_cuda_auto_fxx_on_non_mechanical_records(which, batch):
    """RBT_FXX_AUTO on records whose structural rows are perturbed == the oracle; forcing RBT_FXX_MECHANICAL on the same records
    is measurably wrong, so the perturbation does reach the rows the mechanical instance skips."""
    L = Layout(ANYMAL)
    td, ev, ctrl = FXX_SCHEDULES[which]()
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=batch, seed=71 + batch)
    kkt = _non_mechanical(L, ctrl, kkt, 72 + batch)
    ref = _oracle(L, ctrl, kkt, dx0)
    _assert_oracle(L, ctrl, _solve(ctrl, kkt, dx0, FXX_AUTO), ref)
    _assert_oracle(L, ctrl, _solve(ctrl, kkt, dx0, FXX_GENERAL), ref)
    assert _deviation(L, ctrl, _solve(ctrl, kkt, dx0, FXX_MECHANICAL), ref) > 1e-6


def _single_entry_cases(ctrl, batch):
    """(name, OCP, grid point, row, col, delta): one deviation from the mechanical structure each."""
    nv = ANYMAL.nv
    last = len(ctrl) - 2
    imp = next(i for i, c in enumerate(ctrl) if c.type == IMPACT)
    return [("Fqv[17,17] last grid point, last OCP", batch - 1, last, 17, nv + 17, 0.05),
            ("Fqv[17,17] first grid point, OCP 0", 0, 0, 17, nv + 17, 0.05),
            ("Fqq[6,10] impact stage", batch // 2, imp, 6, 10, 0.05)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", [0, 1, 2])
def test_cuda_auto_fxx_detects_a_single_deviating_entry(case):
    L = Layout(ANYMAL)
    td, ev, ctrl = crawl_schedule("crawl_small")
    batch = 5
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=batch, seed=81)
    name, b, i, r, c, delta = _single_entry_cases(ctrl, batch)[case]
    kkt[b, i, L.k_Fxx + r + c * ANYMAL.nx] += delta
    ref = _oracle(L, ctrl, kkt, dx0)
    _assert_oracle(L, ctrl, _solve(ctrl, kkt, dx0, FXX_AUTO), ref)
    assert _deviation(L, ctrl, _solve(ctrl, kkt, dx0, FXX_MECHANICAL), ref) > 1e-6, name


@pytest.mark.gpu
def test_cuda_auto_fxx_exempt_floating_base_block():
    """A deviation inside the 6 x 6 floating-base block of Fqq is structural (the mechanical instance reads that block)."""
    L = Layout(ANYMAL)
    td, ev, ctrl = crawl_schedule("crawl_small")
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=3, seed=82)
    kkt[1, 4, L.k_Fxx + 2 + 3 * ANYMAL.nx] += 0.05
    ref = _oracle(L, ctrl, kkt, dx0)
    auto = _solve(ctrl, kkt, dx0, FXX_AUTO)
    _assert_oracle(L, ctrl, auto, ref)
    for a, m in zip(auto, _solve(ctrl, kkt, dx0, FXX_MECHANICAL)):
        np.testing.assert_array_equal(a, m)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["crawl_small", "trot_n40"])
def test_cuda_mechanical_records_auto_equals_mechanical(which):
    L = Layout(ANYMAL)
    td, ev, ctrl = {"crawl_small": lambda: crawl_schedule("crawl_small"), "trot_n40": lambda: trot_schedule(40)}[which]()
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=4, seed=83)
    auto, mech = _solve(ctrl, kkt, dx0, FXX_AUTO), _solve(ctrl, kkt, dx0, FXX_MECHANICAL)
    for a, m in zip(auto, mech):
        np.testing.assert_array_equal(a, m)
    ref = _oracle(L, ctrl, kkt, dx0)
    _assert_oracle(L, ctrl, _solve(ctrl, kkt, dx0, FXX_GENERAL), ref)


@pytest.mark.gpu
def test_cuda_kkt_upload_after_condensing_is_inspected():
    """rbt_condense marks the KKT buffer as mechanical; a later rbt_upload(RBT_BUF_KKT) of non-mechanical records must clear
    that, so the next backward sweep checks the records again."""
    from robotoc_b200 import DirectMultipleShooting, RiccatiRecursion, StageDims, StageLayout, anymal_constraint_table
    from synth import make_stage_inputs
    L = Layout(ANYMAL)
    td, ev, ctrl = crawl_schedule("crawl_small")
    batch = 3
    table = anymal_constraint_table()
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S = StageLayout(sd)
    lin, con, sol, dx0s = make_stage_inputs(sd, S, ctrl, batch, 84)
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=batch, seed=85)
    kkt = _non_mechanical(L, ctrl, kkt, 86)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), batch)
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    dms.condense(lin, con)
    rr.backwardRiccatiRecursion(kkt, write_fact=True)
    rr.forwardRiccatiRecursion(dx0)
    got = rr.getRiccatiFactorization(), rr.getDirection(), rr.getFactorizedKKT()
    assert int(rr.info().max()) == 0
    rr.close()
    _assert_oracle(L, ctrl, got, _oracle(L, ctrl, kkt, dx0))
