"""Golden fixtures (tests/golden/golden_r1.npz, made by tests/golden/make_golden.py from the pinned oracle):
CPU: the oracle still reproduces them;  GPU: the CUDA path reproduces them through the C ABI."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import golden_io  # noqa: E402
import make_golden as mg  # noqa: E402

G = golden_io.load(os.path.join(HERE, "golden", "golden_r1.npz"))


def _close(a, b, tol):
    """Over the entries the fixture holds (golden_io)."""
    m = golden_io.finite(b)
    s = np.max(np.abs(b[m]))
    return np.max(np.abs(a[m] - b[m])) <= tol * max(s, 1e-300)


def test_oracle_reproduces_golden():
    ric, d = mg.riccati_case(False)
    assert _close(ric, G["ric"], 1e-12) and _close(d, G["d"], 1e-12)
    ric, d = mg.riccati_case(True)
    assert _close(ric, G["ric_sto"], 1e-12) and _close(d, G["d_sto"], 1e-12)
    ric, d = mg.unconstr_case()
    assert _close(ric, G["uric"], 1e-12) and _close(d, G["ud"], 1e-12)
    kkt_c, steps, sol, con = mg.iteration_case()
    assert _close(kkt_c, G["kkt_condensed"], 1e-12) and _close(steps, G["steps"], 1e-12)
    assert _close(sol, G["sol"], 1e-12) and _close(con, G["con"], 1e-12)
    kkt_c, steps, sol, con = mg.iteration_case(True)
    assert _close(kkt_c, G["kkt_condensed_sto"], 1e-12) and _close(steps, G["steps_sto"], 1e-12)
    assert _close(sol, G["sol_sto"], 1e-12) and _close(con, G["con_sto"], 1e-12)
    ukkt, usteps, usol, ucon = mg.unconstr_iteration_case()
    assert _close(ukkt, G["ukkt_condensed"], 1e-12) and _close(usteps, G["usteps"], 1e-12)
    assert _close(usol, G["usol"], 1e-12) and _close(ucon, G["ucon"], 1e-12)


@pytest.mark.gpu
def test_cuda_reproduces_golden():
    from helpers import small_event_schedule
    from robotoc_b200 import (ANYMAL, DirectMultipleShooting, Layout, RiccatiRecursion, StageDims, StageLayout, ULayout,
                              UnconstrRiccatiRecursion, anymal_constraint_table)
    from synth import make_stage_inputs
    from synth import make_kkt, make_unconstr_kkt
    L = Layout(ANYMAL)
    for sto, kr, kd in ((False, "ric", "d"), (True, "ric_sto", "d_sto")):
        td, ev, ctrl = small_event_schedule(sto)
        kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=2, seed=mg.SEEDS["riccati_sto" if sto else "riccati"])
        rr = RiccatiRecursion(ANYMAL, len(ctrl), 2)
        rr.setTimeDiscretization(ctrl)
        ric, d = rr.solve_host(kkt, dx0)
        # P, s, K, k and the Newton direction (north_star: 1e-6 relative; asserted 1e-8)
        core = slice(0, L.r_core_size)
        assert _close(ric[..., core], G[kr][..., core], 1e-8) and _close(d, G[kd], 1e-8)
        rr.close()
    UL = ULayout(7)
    kkt, dx0 = make_unconstr_kkt(7, UL, 20, 2, mg.SEEDS["unconstr"])
    ur = UnconstrRiccatiRecursion(7, 20, 0.05, 2)
    ric, d = ur.solve_host(kkt, dx0)
    assert _close(ric, G["uric"], 1e-8) and _close(d, G["ud"], 1e-8)
    ur.close()
    table = anymal_constraint_table()
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=4, n_box=table.n_box)
    S = StageLayout(sd)
    for sto, sfx in ((False, ""), (True, "_sto")):
        td, ev, ctrl = small_event_schedule(sto)
        lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, 2, mg.SEEDS["iteration_sto" if sto else "iteration"])
        rr = RiccatiRecursion(ANYMAL, len(ctrl), 2)
        rr.setTimeDiscretization(ctrl)
        dms = DirectMultipleShooting(rr, sd, table)
        dms.condense(lin, con)
        from iteration_check import mask_unread_sto  # hx, hu, h, Qtt exist only where the phase duration is optimised
        K = Layout(ANYMAL)
        assert _close(mask_unread_sto(K, S, ctrl, kkt=dms.getKKT()), mask_unread_sto(K, S, ctrl, kkt=np.array(G["kkt_condensed" + sfx])), 1e-8)
        rr.backwardRiccatiRecursion()
        rr.forwardRiccatiRecursion(dx0)
        dms.computeStepSizes()
        dms.integrateSolution(sol)
        steps = np.stack([dms.maxPrimalStepSize(), dms.maxDualStepSize()], axis=1)
        assert _close(steps, G["steps" + sfx], 1e-10)
        assert _close(dms.getSolution(), G["sol" + sfx], 1e-8)
        rr.close()
    # unconstrained full iteration (iiwa14)
    from robotoc_b200 import UnconstrDirectMultipleShooting, iiwa14_constraint_table
    from synth import make_unconstr_stage_inputs
    tab = iiwa14_constraint_table()
    ur = UnconstrRiccatiRecursion(7, 20, 0.05, 2)
    udms = UnconstrDirectMultipleShooting(ur, tab)
    lin, con, sol, dx0 = make_unconstr_stage_inputs(udms.layout, 20, 2, mg.SEEDS["unconstr_iteration"])
    sol2, con2, steps2 = udms.iteration_host(lin, con, sol, dx0)
    assert _close(udms.getKKT(), G["ukkt_condensed"], 1e-9)
    assert _close(steps2, G["usteps"], 1e-10) and _close(sol2, G["usol"], 1e-9) and _close(con2, G["ucon"], 1e-9)
    ur.close()
