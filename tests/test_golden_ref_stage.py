"""The stage layer (condensing, expansion, step sizes, slack / dual update: SURVEY.md 8a rows a10-a16) pinned against the
reference's own code.  tests/golden/golden_ref_stage_r2.npz holds one full iteration computed by the reference's sources, and
golden_ref_stage_seed_*.npz the same records for further schedules and seeds (make_golden_ref_stage.py);
  CPU: the oracle reproduces them, and the PerformanceIndex the reference's evalKKT members compute;
  GPU: the CUDA path reproduces the full iteration through the C ABI."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import golden_io  # noqa: E402
import make_golden_ref_stage as mg  # noqa: E402

import oracle_lib  # noqa: E402
from iteration_check import mask_unread_sto, oracle_iteration, reference_view_of_expansion  # noqa: E402
from robotoc_b200.grid import IMPACT, TERMINAL  # noqa: E402

G = golden_io.load(os.path.join(HERE, "golden", "golden_ref_stage_r2.npz"))
TOL = 1e-10


def _cmp_records(S, K, ctrl, got, ref, tol, skip_sol=True, impact_cones=False):
    """Every section the reference's code produces, stage by stage (sections it leaves untouched are not compared)."""
    def rel(name, a, b):
        m = golden_io.finite(b)  # the entries the fixture holds
        assert m.all() or np.any(b[m]), f"{name}: the fixture holds none of the section's non-zeros"
        a, b = a[m], b[m]
        s = float(np.max(np.abs(b)))
        if s == 0.0:
            assert float(np.max(np.abs(a))) == 0.0, name
            return
        e = float(np.max(np.abs(a - b))) / s
        assert e < tol, f"{name}: {e:.2e}"
    nx, nu, nv = K.nx, K.nu, K.nv
    got, ref = dict(got), dict(ref)
    for dct in (got, ref):  # sections nothing reads on grid points without switching-time optimisation
        dct["kkt"] = mask_unread_sto(K, S, ctrl, kkt=np.array(dct["kkt"]))
        dct["ex_upd"] = mask_unread_sto(K, S, ctrl, ex=np.array(dct["ex_upd"]))
    for i, c in enumerate(ctrl):
        rel(f"Qxx[{i}]", got["kkt"][:, i, K.k_Qxx:K.k_Qxx + nx * nx], ref["kkt"][:, i, K.k_Qxx:K.k_Qxx + nx * nx])
        rel(f"lx[{i}]", got["kkt"][:, i, K.k_lx:K.k_lx + nx], ref["kkt"][:, i, K.k_lx:K.k_lx + nx])
        rel(f"P[{i}]", got["ric"][:, i, K.r_P:K.r_P + nx * nx], ref["ric"][:, i, K.r_P:K.r_P + nx * nx])
        rel(f"dx[{i}]", got["d_upd"][:, i, K.d_dx:K.d_dx + nx], ref["d_upd"][:, i, K.d_dx:K.d_dx + nx])
        rel(f"dlmdgmm[{i}]", got["d_upd"][:, i, K.d_dlmdgmm:K.d_dlmdgmm + nx], ref["d_upd"][:, i, K.d_dlmdgmm:K.d_dlmdgmm + nx])
        if c.type == TERMINAL:
            continue
        nvf = nv + c.nf
        rel(f"kkt[{i}]", got["kkt"][:, i], ref["kkt"][:, i])
        for f, n in (("e_Z", S.nvf * S.nvf), ("e_R", S.nvf * nx), ("e_r", nvf), ("e_Qafqv", S.nvf * nx), ("e_laf", nvf), ("e_Fqqpi", 36)):
            o = getattr(S, f)
            rel(f"{f}[{i}]", got["ex_upd"][:, i, o:o + n], ref["ex_upd"][:, i, o:o + n])
        rel(f"daf[{i}]", got["xd_exp"][:, i, S.x_daf:S.x_daf + nvf], ref["xd_exp"][:, i, S.x_daf:S.x_daf + nvf])
        rel(f"dbetamu[{i}]", got["xd_upd"][:, i, S.x_dbetamu:S.x_dbetamu + nvf], ref["xd_upd"][:, i, S.x_dbetamu:S.x_dbetamu + nvf])
        if c.type == IMPACT:
            if impact_cones:  # the ImpactFrictionCone rows (the box rows do not exist on an impact stage)
                for key, fields in (("cc_cond", ("c_cmpl", "c_cond")), ("cc_exp", ("c_dslack", "c_ddual")), ("cc_upd", ("c_slack", "c_dual"))):
                    for f in fields:
                        o = getattr(S, f)
                        rel(f"impact {f}[{i}]", got[key][:, i, o + S.nbox:o + S.nc], ref[key][:, i, o + S.nbox:o + S.nc])
            continue
        for f, n in (("e_Qafu", S.nvf * nv), ("e_Qxup", nx * S.np), ("e_Quup", S.np * nu), ("e_lup", S.np), ("e_haf", nvf)):
            o = getattr(S, f)
            rel(f"{f}[{i}]", got["ex_upd"][:, i, o:o + n], ref["ex_upd"][:, i, o:o + n])
        rel(f"dnup[{i}]", got["xd_upd"][:, i, S.x_dnup:S.x_dnup + S.np], ref["xd_upd"][:, i, S.x_dnup:S.x_dnup + S.np])
        rel(f"K[{i}]", got["ric"][:, i, K.r_K:K.r_K + nx * nu], ref["ric"][:, i, K.r_K:K.r_K + nx * nu])
        rel(f"du[{i}]", got["d_upd"][:, i, K.d_du:K.d_du + nu], ref["d_upd"][:, i, K.d_du:K.d_du + nu])
        for key, fields in (("cc_cond", ("c_cmpl", "c_cond")), ("cc_exp", ("c_dslack", "c_ddual")), ("cc_upd", ("c_slack", "c_dual"))):
            for f in fields:
                o = getattr(S, f)
                rel(f"{f}[{i}]", got[key][:, i, o:o + S.nc], ref[key][:, i, o:o + S.nc])
    rel("steps", got["steps"], ref["steps"])


@pytest.mark.parametrize("impact_cones", [False, True])
def test_oracle_reproduces_the_reference_iteration_golden(impact_cones):
    lib = oracle_lib.load()
    table, sd, S, K, ctrl, lin, con, sol, dx0 = mg.problem(lib.orc_stage_layout_get, lib.orc_layout_get, impact_cones)
    got = oracle_iteration(sd, S, K, table, ctrl, lin, con, sol, dx0)
    ref = {k[3:]: G[k] for k in G if k.startswith("ic_")} if impact_cones else G
    if impact_cones:  # the impact cones must matter: the iteration differs from the one without them
        assert np.nanmax(np.abs(ref["ric"] - G["ric"])) > 1e-6 and abs(float(ref["steps"][0, 0]) - float(G["steps"][0, 0])) >= 0.0
    _cmp_records(S, K, ctrl, got, ref, TOL, impact_cones=impact_cones)


def _oracle_perf_stage(lib, sd, S, table, ctrl, lin, con):
    """orc_stage_perf_index per grid point: {cost_barrier, primal_feasibility, dual_feasibility, kkt_error}."""
    import ctypes
    lib.orc_stage_perf_index.argtypes = [ctypes.c_void_p] * 6
    out = np.zeros((lin.shape[0], len(ctrl), 4))
    csd = sd.c()
    for b in range(lin.shape[0]):
        for i, c in enumerate(ctrl):
            st = np.zeros(4)
            lib.orc_stage_perf_index(ctypes.byref(csd), ctypes.byref(table), ctypes.byref(c), oracle_lib.ptr(np.ascontiguousarray(lin[b, i])),
                                     oracle_lib.ptr(np.ascontiguousarray(con[b, i])), oracle_lib.ptr(st))
            out[b, i] = st
    return out


@pytest.mark.parametrize("impact_cones", [False, True])
def test_oracle_performance_index_equals_the_reference_evalKKT_summary(impact_cones):
    """PerformanceIndex of every grid point (log barrier, primal / dual feasibility, squared KKT error) as the reference's own
    members compute it before condensing (OCPData / SplitKKTResidual / ConstraintsData / ContactDynamicsData ::KKTError etc.,
    intermediate_stage.cpp:124-132, impact_stage.cpp:104-113, terminal_stage.cpp:94-100) -- on the small event schedule and
    on the BASELINE trot schedule."""
    lib = oracle_lib.load()
    table, sd, S, K, ctrl, lin, con, sol, dx0 = mg.problem(lib.orc_stage_layout_get, lib.orc_layout_get, impact_cones)
    got = _oracle_perf_stage(lib, sd, S, table, ctrl, lin, con)
    ref = G["ic_perf_stage" if impact_cones else "perf_stage"]
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-300)
    assert (ref[:, :, 3] > 0).all() and (ref[:, :-1, 0] != 0).any()
    table, sd, S, K, ctrl, lin, con, sol, dx0 = mg.perf_trot_problem(impact_cones, lib.orc_stage_layout_get, lib.orc_layout_get)
    np.testing.assert_allclose(_oracle_perf_stage(lib, sd, S, table, ctrl, lin, con), G[f"perf_trot_{int(impact_cones)}"],
                               rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("which,seed", list(mg.SEED_CASES.items()))
def test_oracle_equals_live_reference_stage_layer(which, seed):
    lib = oracle_lib.load()
    table, sd, S, K, ctrl, lin, con, sol, dx0 = mg.seed_problem(which, seed, lib.orc_stage_layout_get, lib.orc_layout_get)
    ref = golden_io.load(mg.seed_path(which))
    got = oracle_iteration(sd, S, K, table, ctrl, lin, con, sol, dx0)
    _cmp_records(S, K, ctrl, got, ref, TOL, impact_cones=which.endswith("_icone"))


@pytest.mark.gpu
@pytest.mark.parametrize("impact_cones", [False, True])
def test_cuda_reproduces_the_reference_iteration_golden(impact_cones):
    from robotoc_b200 import ANYMAL, DirectMultipleShooting, RiccatiRecursion
    table, sd, S, K, ctrl, lin, con, sol, dx0 = mg.problem(impact_cones=impact_cones)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), lin.shape[0])
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, sd, table)
    # PerformanceIndex of evalKKT: {cost (not on this path), barrier, primal / dual feasibility, KKT error, sqrt} vs the reference's sums
    perf = dms.evalKKT(lin, con)
    pref = (G["ic_perf_stage"] if impact_cones else G["perf_stage"]).sum(axis=1)
    np.testing.assert_allclose(perf[:, 1:5], pref, rtol=1e-11)
    np.testing.assert_allclose(perf[:, 5], np.sqrt(pref[:, 3]), rtol=1e-11)
    dms.condense(lin, con)
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
    ref = {k[3:]: G[k] for k in G if k.startswith("ic_")} if impact_cones else G
    _cmp_records(S, K, ctrl, got, ref, 1e-8, impact_cones=impact_cones)
    rr.close()
