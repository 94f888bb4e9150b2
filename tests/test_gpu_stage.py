"""GPU parity of the stage layer (rows a10-a16) and of a full hot-path iteration
condense -> backward -> forward -> step sizes -> update, against the CPU oracle, through the C ABI."""
import ctypes

import os

import numpy as np
import pytest

import oracle_lib
from helpers import jump_sto_schedule, rel_err, small_event_schedule, trot_schedule
from robotoc_b200 import ANYMAL, DirectMultipleShooting, Layout, RiccatiRecursion, StageDims, StageLayout, anymal_constraint_table
from robotoc_b200.grid import IMPACT, TERMINAL
from synth import make_stage_inputs, robotoc_cost_structure, symmetrize_lin

pytestmark = pytest.mark.gpu
TOL = 1e-8


def _oracle_iteration(lib, sd, S, K, table, ctrl, lin, con, sol, dx0):
    batch, n_grid = lin.shape[0], lin.shape[1]
    csd = sd.c()
    kkt = np.zeros((batch, n_grid, K.k_stride))
    ex = np.zeros((batch, n_grid, S.e_stride))
    cc, ss = con.copy(), sol.copy()
    assert lib.orc_condense_batch(ctypes.byref(csd), ctypes.byref(table), ctrl, n_grid, batch, oracle_lib.ptr(lin),
                                  oracle_lib.ptr(cc), oracle_lib.ptr(kkt), oracle_lib.ptr(ex), 0) == 0
    cc_after_condense = cc.copy()
    kk, ric, d, info = oracle_lib.riccati_batch(ANYMAL, K, ctrl, kkt, dx0)
    assert info == 0
    xd = np.zeros((batch, n_grid, S.x_stride))
    steps = np.zeros((batch, 2))
    lib.orc_expand_batch(ctypes.byref(csd), ctypes.byref(table), ctrl, n_grid, batch, oracle_lib.ptr(lin), oracle_lib.ptr(ex),
                         oracle_lib.ptr(d), oracle_lib.ptr(cc), oracle_lib.ptr(xd), oracle_lib.ptr(steps), 0)
    d_before, cc_after_expand, xd_after_expand = d.copy(), cc.copy(), xd.copy()
    lib.orc_update_batch(ctypes.byref(csd), ctypes.byref(table), ctrl, n_grid, batch, oracle_lib.ptr(ex), oracle_lib.ptr(d),
                         oracle_lib.ptr(xd), oracle_lib.ptr(cc), oracle_lib.ptr(ss), oracle_lib.ptr(steps), 0)
    return dict(kkt=kkt, ex0=None, cc_cond=cc_after_condense, ric=ric, d=d_before, cc_exp=cc_after_expand, xd_exp=xd_after_expand,
                steps=steps, d_upd=d, xd_upd=xd, cc_upd=cc, sol=ss, ex_upd=ex)


def _cmp(name, got, ref, tol=TOL):
    scale = np.max(np.abs(ref))
    if scale == 0.0:
        assert np.max(np.abs(got)) == 0.0, f"{name}: expected zeros"
        return
    e = np.max(np.abs(got - ref)) / scale
    assert e < tol, f"{name}: rel err {e:.3e}"


def _cmp_rows(name, S, c, icone, f, got, ref):
    """PDIPM rows of one stage: all rows on Intermediate / Lift stages, the ImpactFrictionCone rows on Impact stages."""
    o = getattr(S, f)
    if c.type == IMPACT:
        if icone:
            _cmp(name, got[:, o + S.nbox:o + S.nc], ref[:, o + S.nbox:o + S.nc])
    else:
        _cmp(name, got[:, o:o + S.nc], ref[:, o:o + S.nc])


def poison_inactive_contact_rows(S, ctrl, lin):
    """A copy of the linearization records with NaN in the rows nf..nf_max-1 of every contact Jacobian J: rows no kernel may
    use (a record reused from a phase with more contacts, or left by the wire format, which never writes them)."""
    out = lin.copy()
    for i, c in enumerate(ctrl):
        if c.type != TERMINAL:
            J = out[:, i, S.l_J:S.l_J + S.nfm * S.nv].reshape(-1, S.nv, S.nfm)  # [batch, col, row]
            J[:, :, c.nf:] = np.nan
    return out


def _run(ctrl, batch, seed, reserve=0, impact_cones=False, poison=False):
    """poison: the device gets the records with NaN in the inactive rows of J (poison_inactive_contact_rows)."""
    lib = oracle_lib.load()
    table = anymal_constraint_table(impact_friction_cone=impact_cones)
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S, K = StageLayout(sd), Layout(ANYMAL)
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, batch, seed, impact_cones=impact_cones)
    ref = _oracle_iteration(lib, sd, S, K, table, ctrl, lin, con, sol, dx0)
    if poison:
        lin = poison_inactive_contact_rows(S, ctrl, lin)
    rr = RiccatiRecursion(ANYMAL, len(ctrl) + reserve, batch)  # reserve: the reference sizes for N + 1 + reserved events
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    dms.condense(lin, con)
    kkt, cc = dms.getKKT(), dms.getConstraintData()
    assert int(rr.info().max()) == 0
    from iteration_check import mask_unread_sto
    kkt, kkt_ref = mask_unread_sto(K, S, ctrl, kkt=kkt), mask_unread_sto(K, S, ctrl, kkt=ref["kkt"].copy())
    for i, c in enumerate(ctrl):
        _cmp(f"kkt[{i}]", kkt[:, i], kkt_ref[:, i])
        if c.type != TERMINAL:
            for f in ("c_cmpl", "c_cond"):
                _cmp_rows(f"{f}[{i}]", S, c, impact_cones, f, cc[:, i], ref["cc_cond"][:, i])
    rr.backwardRiccatiRecursion()
    rr.forwardRiccatiRecursion(dx0)
    d = rr.getDirection()
    _cmp("direction", d, ref["d"])
    dms.computeStepSizes()
    steps = np.stack([dms.maxPrimalStepSize(), dms.maxDualStepSize()], axis=1)
    _cmp("steps", steps, ref["steps"], 1e-10)
    xd, cc = dms.getExpandedDirection(), dms.getConstraintData()
    for i, c in enumerate(ctrl):
        if c.type == TERMINAL:
            continue
        _cmp(f"daf[{i}]", xd[:, i, S.x_daf:S.x_daf + 18 + c.nf], ref["xd_exp"][:, i, S.x_daf:S.x_daf + 18 + c.nf])
        for f in ("c_dslack", "c_ddual"):
            _cmp_rows(f"{f}[{i}]", S, c, impact_cones, f, cc[:, i], ref["cc_exp"][:, i])
    dms.integrateSolution(sol)
    sol_g, cc, xd, d2 = dms.getSolution(), dms.getConstraintData(), dms.getExpandedDirection(), rr.getDirection()
    for i, c in enumerate(ctrl):
        _cmp(f"sol[{i}]", sol_g[:, i], ref["sol"][:, i])
        _cmp(f"dlmdgmm[{i}]", d2[:, i, K.d_dlmdgmm:K.d_dlmdgmm + 36], ref["d_upd"][:, i, K.d_dlmdgmm:K.d_dlmdgmm + 36])
        if c.type != TERMINAL:
            _cmp(f"dbetamu[{i}]", xd[:, i, S.x_dbetamu:S.x_dbetamu + 18 + c.nf], ref["xd_upd"][:, i, S.x_dbetamu:S.x_dbetamu + 18 + c.nf])
            if c.type != IMPACT:
                _cmp(f"dnup[{i}]", xd[:, i, S.x_dnup:S.x_dnup + 6], ref["xd_upd"][:, i, S.x_dnup:S.x_dnup + 6])
            for f in ("c_slack", "c_dual"):
                _cmp_rows(f"{f}[{i}]", S, c, impact_cones, f, cc[:, i], ref["cc_upd"][:, i])
    from iteration_check import reference_view_of_expansion
    ex = reference_view_of_expansion(S, dms.getExpansionData())  # full Qafqv / Qafu from the contact rows + diag(Qaa) kept on the device
    for i, c in enumerate(ctrl):
        if c.type != TERMINAL:
            nz = 1080 if c.type == IMPACT else 1080 + 540  # Qafqv | Qafu (Qafu does not exist on an impact stage)
            _cmp(f"Qafqv|Qafu[{i}]", ex[:, i, S.e_Qafqv:S.e_Qafqv + nz], ref["ex_upd"][:, i, S.e_Qafqv:S.e_Qafqv + nz])
            for f, n in (("e_Z", 900), ("e_R", 1080), ("e_r", 30), ("e_laf", 30)):
                o = getattr(S, f)
                _cmp(f"{f}[{i}]", ex[:, i, o:o + n], ref["ex_upd"][:, i, o:o + n])
    # the one-call host path (chunked, trimmed transfers) gives the same bits as the step-by-step path
    for chunks in ("1", "3"):
        os.environ["RBT_E2E_CHUNKS"] = chunks
        sol2, con2, steps2 = dms.iteration_host(lin, con, sol, dx0)
        used = S.s_xi + S.nsm
        np.testing.assert_array_equal(sol2[:, :, :used], sol_g[:, :, :used])
        np.testing.assert_array_equal(steps2, steps)
        for f in ("c_slack", "c_dual"):
            o = getattr(S, f)
            np.testing.assert_array_equal(con2[:, :, o:o + S.nc], cc[:, :, o:o + S.nc])
        np.testing.assert_array_equal(con2[:, :, S.c_res:], con[:, :, S.c_res:])  # not refreshed from the device
    del os.environ["RBT_E2E_CHUNKS"]
    h2d, d2h = dms.iteration_host_bytes()
    assert 0 < d2h < h2d < lin.nbytes + con.nbytes + sol.nbytes + dx0.nbytes
    # host wire format (packed symmetric blocks): same bits as the classic records once those are exactly symmetric
    lin_s = symmetrize_lin(S, lin)
    sol3, con3, steps3 = dms.iteration_host(lin_s, con, sol, dx0)
    sol4, con4, steps4 = dms.iteration_host_wire(dms.pack_wire(lin_s), lin_s, con, sol, dx0)
    np.testing.assert_array_equal(sol4, sol3)
    np.testing.assert_array_equal(con4, con3)
    np.testing.assert_array_equal(steps4, steps3)
    assert rel_err(sol3[:, :, :used], sol_g[:, :, :used]) < 1e-9  # symmetrising moves the inputs by rounding only
    assert dms.iteration_host_bytes(wire=True)[0] < 0.80 * h2d
    # resident solver state: solution, slack and dual stay on the device, only wire records + residuals + dx0 go up
    dms.setSolution(sol)
    dms.setConstraintData(con)
    res = np.ascontiguousarray(con[:, :, S.c_res:S.c_res + S.ncp])
    sol5, sd5, steps5 = dms.iteration_host_resident(dms.pack_wire(lin_s), lin_s, res, dx0)
    np.testing.assert_array_equal(sol5[:, :, :used], sol3[:, :, :used])
    np.testing.assert_array_equal(steps5, steps3)
    np.testing.assert_array_equal(sd5[:, :, :S.nc], con3[:, :, S.c_slack:S.c_slack + S.nc])
    np.testing.assert_array_equal(sd5[:, :, S.ncp:S.ncp + S.nc], con3[:, :, S.c_dual:S.c_dual + S.nc])
    assert dms.iteration_host_bytes(resident=True)[0] < 0.90 * dms.iteration_host_bytes(wire=True)[0]
    # ... and a second resident iteration continues from the updated state (what a host-driven SQP loop does)
    sol6, sd6, steps6 = dms.iteration_host_resident(dms.pack_wire(lin_s), lin_s, res, dx0)
    con_b = con3.copy()
    con_b[:, :, S.c_res:S.c_res + S.ncp] = res
    sol7, con7, steps7 = dms.iteration_host_wire(dms.pack_wire(lin_s), lin_s, con_b, sol3, dx0)
    np.testing.assert_array_equal(sol6[:, :, :used], sol7[:, :, :used])
    np.testing.assert_array_equal(steps6, steps7)
    # wire records with robotoc's cost structure (Qqq dense, Qvv / Quu / Qff diagonal): same bits as the dense records
    lin_c = robotoc_cost_structure(S, lin)
    sol8, con8, steps8 = dms.iteration_host(lin_c, con, sol, dx0)
    w_gen = dms.pack_wire(lin_c)
    dms.setWireCostStructure(True)
    w_rob = dms.pack_wire(lin_c)
    assert w_rob.shape[1] < 0.82 * w_gen.shape[1]
    sol9, con9, steps9 = dms.iteration_host_wire(w_rob, lin_c, con, sol, dx0)
    dms.setWireCostStructure(False)
    np.testing.assert_array_equal(sol9, sol8)
    np.testing.assert_array_equal(con9, con8)
    np.testing.assert_array_equal(steps9, steps8)
    rr.close()


def test_stage_layer_small_event_schedule():
    td, ev, ctrl = small_event_schedule(False)
    _run(ctrl, batch=3, seed=21)


def test_stage_layer_trot_n40():
    td, ev, ctrl = trot_schedule(40)
    _run(ctrl, batch=2, seed=22)


def test_stage_layer_impact_friction_cones():
    """ImpactFrictionCone registered (examples/anymal/run.cpp:173-181): the Impact stages carry cone rows on the impact forces
    -- condensing into Qqq / Qqf / Qff / lq / lf, slack / dual directions, step sizes, update (impact_friction_cone.cpp)."""
    td, ev, ctrl = small_event_schedule(True)
    assert any(c.type == IMPACT for c in ctrl)
    _run(ctrl, batch=3, seed=26, impact_cones=True)
    td, ev, ctrl = trot_schedule(40)
    _run(ctrl, batch=2, seed=27, impact_cones=True)


def test_stage_layer_small_event_schedule_sto():
    """Switching-time optimisation on: hx / hu / fx / Qtt scaling in the condensing, dts terms in the dual expansion."""
    td, ev, ctrl = small_event_schedule(True)
    _run(ctrl, batch=3, seed=23)


def test_stage_layer_jump_sto_n80():
    """BASELINE.json configs[3] schedule (ANYmal jumping, STO, N=80) through the full iteration."""
    td, ev, ctrl = jump_sto_schedule(80)
    _run(ctrl, batch=2, seed=24)


def test_stage_layer_single_ocp_with_reserved_grid_points():
    """batch = 1 (the reference's own use) on a handle sized for more grid points than the schedule has
    (riccati_recursion.cpp:12-13: N + 1 + reserved_num_discrete_events)."""
    td, ev, ctrl = small_event_schedule(False)
    _run(ctrl, batch=1, seed=25, reserve=4)
