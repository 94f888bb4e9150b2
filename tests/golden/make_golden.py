"""Generates the golden fixtures under tests/golden/ from the CPU oracle (oracle/*.c) on fixed-seed inputs.

    python tests/golden/make_golden.py

The reference itself (Eigen3 + Pinocchio C++) cannot be built or imported in this image, and its test-suite holds no
golden vectors (SURVEY.md section 4), so these fixtures pin the ORACLE (regression) and give the GPU tests a
size-independent, file-based target; the oracle in turn is pinned by the identity tests (test_oracle_kkt.py,
test_oracle_condense.py).  Inputs are regenerated from the seeds below by the tests; only outputs are stored, sampled by
golden_io.
"""
import ctypes
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_lib  # noqa: E402
from helpers import small_event_schedule  # noqa: E402
from robotoc_b200 import ANYMAL, Layout, ULayout  # noqa: E402
from robotoc_b200.stage import StageDims, StageLayout, anymal_constraint_table  # noqa: E402
from synth import make_stage_inputs  # noqa: E402
from synth import make_kkt, make_unconstr_kkt  # noqa: E402

SEEDS = {"riccati": 101, "riccati_sto": 102, "unconstr": 103, "iteration": 104, "iteration_sto": 105, "unconstr_iteration": 106}


def riccati_case(sto):
    lib = oracle_lib.load()
    L = Layout(ANYMAL, getter=lib.orc_layout_get)
    td, ev, ctrl = small_event_schedule(sto)
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=2, seed=SEEDS["riccati_sto" if sto else "riccati"])
    kk, ric, d, info = oracle_lib.riccati_batch(ANYMAL, L, ctrl, kkt, dx0)
    assert info == 0
    return ric, d


def unconstr_case():
    lib = oracle_lib.load()
    UL = ULayout(7, getter=lib.orc_ulayout_get)
    kkt, dx0 = make_unconstr_kkt(7, UL, 20, 2, SEEDS["unconstr"])
    kk, ric, d, info = oracle_lib.unconstr_batch(7, UL, 20, 0.05, kkt, dx0)
    assert info == 0
    return ric, d


def unconstr_iteration_case():
    """Full unconstrained iteration (iiwa14, N=20, batch 2): condense -> Riccati -> step sizes -> update."""
    from robotoc_b200.unconstr_dms import UStageLayout, iiwa14_constraint_table
    from synth import make_unconstr_stage_inputs
    lib = oracle_lib.load()
    tab = iiwa14_constraint_table()
    S = UStageLayout(7, tab.n_box, getter=lib.orc_ustage_layout_get)
    UL = ULayout(7, getter=lib.orc_ulayout_get)
    lin, con, sol, dx0 = make_unconstr_stage_inputs(S, 20, 2, SEEDS["unconstr_iteration"])
    out = oracle_lib.unconstr_iteration(7, UL, S, tab, 20, 0.05, lin, con, sol, dx0)
    assert out["info"] == 0
    return out["kkt"], out["steps"], out["sol"], out["con"]


def iteration_case(sto=False):
    lib = oracle_lib.load()
    table = anymal_constraint_table()
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=4, n_box=table.n_box)
    S = StageLayout(sd, getter=lib.orc_stage_layout_get)
    K = Layout(ANYMAL, getter=lib.orc_layout_get)
    td, ev, ctrl = small_event_schedule(sto)
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, 2, SEEDS["iteration_sto" if sto else "iteration"])
    n_grid, batch = len(ctrl), 2
    csd = sd.c()
    kkt, ex = np.zeros((batch, n_grid, K.k_stride)), np.zeros((batch, n_grid, S.e_stride))
    P = oracle_lib.ptr
    assert lib.orc_condense_batch(ctypes.byref(csd), ctypes.byref(table), ctrl, n_grid, batch, P(lin), P(con), P(kkt), P(ex), 1) == 0
    kkt_condensed = kkt.copy()
    kk, ric, d, info = oracle_lib.riccati_batch(ANYMAL, K, ctrl, kkt, dx0)
    xd, steps = np.zeros((batch, n_grid, S.x_stride)), np.zeros((batch, 2))
    lib.orc_expand_batch(ctypes.byref(csd), ctypes.byref(table), ctrl, n_grid, batch, P(lin), P(ex), P(d), P(con), P(xd), P(steps), 1)
    lib.orc_update_batch(ctypes.byref(csd), ctypes.byref(table), ctrl, n_grid, batch, P(ex), P(d), P(xd), P(con), P(sol), P(steps), 1)
    return kkt_condensed, steps, sol, con


if __name__ == "__main__":
    ric, d = riccati_case(False)
    ric_s, d_s = riccati_case(True)
    uric, ud = unconstr_case()
    kkt_c, steps, sol, con = iteration_case()
    kkt_cs, steps_s, sol_s, con_s = iteration_case(True)
    ukkt, usteps, usol, ucon = unconstr_iteration_case()
    import golden_io
    from robotoc_b200.unconstr_dms import UStageLayout, iiwa14_constraint_table
    lib = oracle_lib.load()
    K, UL = Layout(ANYMAL, getter=lib.orc_layout_get), ULayout(7, getter=lib.orc_ulayout_get)
    table = anymal_constraint_table()
    S = StageLayout(StageDims(ANYMAL, nf_max=12, n_contacts=4, n_box=table.n_box), getter=lib.orc_stage_layout_get)
    US = UStageLayout(7, iiwa14_constraint_table().n_box, getter=lib.orc_ustage_layout_get)
    data = dict(ric=ric, d=d, ric_sto=ric_s, d_sto=d_s, uric=uric, ud=ud, kkt_condensed=kkt_c, steps=steps, sol=sol, con=con,
                kkt_condensed_sto=kkt_cs, steps_sto=steps_s, sol_sto=sol_s, con_sto=con_s,
                ukkt_condensed=ukkt, usteps=usteps, usol=usol, ucon=ucon)
    layouts = {"ric": (K, "r_"), "d": (K, "d_"), "uric": (UL, "r_"), "ud": (UL, "d_"), "kkt_condensed": (K, "k_"), "sol": (S, "s_"),
               "con": (S, "c_"), "ukkt_condensed": (UL, "k_"), "usol": (US, "s_"), "ucon": (US, "c_")}
    sections = {k: golden_io.sections(*layouts[k.replace("_sto", "")]) for k in data if k.replace("_sto", "") in layouts}
    golden_io.save(os.path.join(HERE, "golden_r1.npz"), data, sections)
    print("wrote", os.path.join(HERE, "golden_r1.npz"), os.path.getsize(os.path.join(HERE, "golden_r1.npz")) // 1024, "KiB")
