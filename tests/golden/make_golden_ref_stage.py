"""Generates tests/golden/golden_ref_stage_r2.npz and golden_ref_stage_seed_<case>.npz: hot-path iterations computed by the reference's own code
(tests/ref_lib.reference_iteration: the reference's src/dynamics, src/constraints, src/core and src/riccati compiled unmodified,
oracle/Makefile.ref).  Only runs where a checkout of the reference is available (ROBOTOC_REFERENCE, see oracle/Makefile.ref):

    python tests/golden/make_golden_ref_stage.py

Stored (sampled by golden_io):
  - one FULL iteration on the small event schedule with switching-time optimisation (Intermediate, Lift,
    switching-constraint and Impact stages), batch 1, without and with impact friction cones ("ic_" keys);
  - golden_ref_stage_seed_<case>.npz: the records tests/test_golden_ref_stage.py compares, for the further schedules / seeds
    of SEED_CASES;
  - "perf_trot_*": the per-grid-point PerformanceIndex of evalKKT on the BASELINE trot schedule (perf_trot_problem());
  - "jl_<case>_*": what the reference's joint position / velocity / torque limit classes add to the gradient and the PDIPM
    residuals (output minus input), for the problems of tests/test_joint_limits.py."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import small_event_schedule, trot_schedule  # noqa: E402
from robotoc_b200 import ANYMAL  # noqa: E402
from robotoc_b200.stage import StageDims, anymal_constraint_table  # noqa: E402
from synth import make_stage_inputs  # noqa: E402

import golden_io  # noqa: E402

SEED, BATCH = 301, 1
KEYS = ("kkt", "cc_cond", "ric", "d", "cc_exp", "xd_exp", "steps", "d_upd", "xd_upd", "cc_upd", "ex_upd", "perf_stage")
SEED_CASES = {"small": 311, "small_sto": 312, "trot": 313, "small_icone": 314, "small_sto_icone": 315}  # name -> seed, batch 1
SEED_KEYS = ("kkt", "cc_cond", "ric", "cc_exp", "xd_exp", "steps", "d_upd", "xd_upd", "cc_upd", "ex_upd")
# the records are compared section by section at every grid point: every grid point keeps the short sections (dx, du, lx, lu,
# e_lup, e_r, ...) whole and at least 36 entries of each longer one
PER_GRID_POINT = dict(block=64, min_keep=36, per_row=True)
JOINT_LIMIT_PROBLEMS = {"small_sto": (lambda: small_event_schedule(True), 2, 81), "trot": (lambda: trot_schedule(40), 2, 81)}  # schedule, batch, seed


def problem(S_getter=None, K_getter=None, impact_cones=False):
    """impact_cones: the same problem with ImpactFrictionCone registered (examples/anymal/run.cpp:173-181): the impact stage
    carries friction-cone rows on the impact forces (golden keys prefixed "ic_")."""
    from robotoc_b200 import Layout, StageLayout
    table = anymal_constraint_table(impact_friction_cone=impact_cones)
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S, K = StageLayout(sd, getter=S_getter), Layout(ANYMAL, getter=K_getter)
    td, ev, ctrl = small_event_schedule(True)
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, BATCH, SEED, impact_cones=impact_cones)
    return table, sd, S, K, ctrl, lin, con, sol, dx0


def seed_problem(which, seed, S_getter=None, K_getter=None):
    from robotoc_b200 import Layout, StageLayout
    icone = which.endswith("_icone")
    table = anymal_constraint_table(impact_friction_cone=icone)
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S, K = StageLayout(sd, getter=S_getter), Layout(ANYMAL, getter=K_getter)
    td, ev, ctrl = {"small": small_event_schedule(False), "small_sto": small_event_schedule(True), "trot": trot_schedule(40),
                    "small_icone": small_event_schedule(False), "small_sto_icone": small_event_schedule(True)}[which]
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, 1, seed, impact_cones=icone)
    return table, sd, S, K, ctrl, lin, con, sol, dx0


def perf_trot_problem(impact_cones, S_getter=None, K_getter=None):
    """BASELINE trot schedule, with switching-constraint residuals that give the primal feasibility something to measure."""
    from robotoc_b200 import Layout, StageLayout
    table = anymal_constraint_table(impact_friction_cone=impact_cones)
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S, K = StageLayout(sd, getter=S_getter), Layout(ANYMAL, getter=K_getter)
    td, ev, ctrl = trot_schedule(40)
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, 1, 316, impact_cones=impact_cones)
    rng = np.random.default_rng(5)
    for i, c in enumerate(ctrl):
        if c.ns > 0:
            lin[:, i, S.l_p:S.l_p + c.ns] = rng.uniform(-1, 1, size=(1, c.ns))
    return table, sd, S, K, ctrl, lin, con, sol, dx0


def joint_limit_problem(sched, batch, seed):
    """A stage problem with joint position / velocity / torque limits of the order of ANYmal's URDF."""
    import ctypes

    import oracle_lib
    from robotoc_b200 import StageLayout
    lib = oracle_lib.load()
    table = anymal_constraint_table()
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S = StageLayout(sd, getter=lib.orc_stage_layout_get)
    td, ev, ctrl = sched
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, batch, seed)
    rng = np.random.default_rng(seed + 3)
    lim = {0: 1.2, 1: 8.0, 3: 40.0}  # |q|, |v|, |u| limits of the order of ANYmal's URDF
    bound = np.array([table.box[r].sign * lim[table.box[r].var] * rng.uniform(0.8, 1.2) for r in range(table.n_box)])
    for k in (2, 4):  # the reference's velocity / torque limits are symmetric (joint_velocity_lower_limit.cpp: vmin = -vmax)
        bound[k * 12:(k + 1) * 12] = -bound[(k + 1) * 12:(k + 2) * 12]
    lib.orc_linearize_joint_limits_batch.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 4
    return lib, table, sd, S, ctrl, lin, con, sol, bound


def seed_path(which):
    return os.path.join(HERE, f"golden_ref_stage_seed_{which}.npz")


def record_sections(S, K, keys):
    """golden_io section offsets of the records this file stores, by key suffix."""
    prefix = {"kkt": (K, "k_"), "ric": (K, "r_"), "d": (K, "d_"), "d_upd": (K, "d_"), "ex_upd": (S, "e_"), "xd_exp": (S, "x_"),
              "xd_upd": (S, "x_"), "cc_cond": (S, "c_"), "cc_exp": (S, "c_"), "cc_upd": (S, "c_"), "dlin": (S, "l_"), "dcon": (S, "c_")}
    out = {}
    for key in keys:
        for suffix, (layout, p) in prefix.items():
            if key.endswith("_" + suffix) or key == suffix:
                out[key] = golden_io.sections(layout, p)
    return out


if __name__ == "__main__":
    import ctypes

    import oracle_lib
    import ref_lib
    lib = oracle_lib.load()
    table, sd, S, K, ctrl, lin, con, sol, dx0 = problem(lib.orc_stage_layout_get, lib.orc_layout_get)
    out = ref_lib.reference_iteration(sd, S, K, table, ctrl, lin, con, dx0)
    data = {k: out[k] for k in KEYS}
    table, sd, S, K, ctrl, lin, con, sol, dx0 = problem(lib.orc_stage_layout_get, lib.orc_layout_get, impact_cones=True)
    out = ref_lib.reference_iteration(sd, S, K, table, ctrl, lin, con, dx0)
    data.update({"ic_" + k: out[k] for k in KEYS})
    for impact_cones in (False, True):
        table, sd, S, K, ctrl, lin, con, sol, dx0 = perf_trot_problem(impact_cones, lib.orc_stage_layout_get, lib.orc_layout_get)
        data[f"perf_trot_{int(impact_cones)}"] = ref_lib.reference_iteration(sd, S, K, table, ctrl, lin, con, dx0)["perf_stage"]
    rl = ref_lib.load()
    rl.ref_linearize_joint_limits.argtypes = [ctypes.c_void_p] * 7
    P = oracle_lib.ptr
    for which, (sched, batch, seed) in JOINT_LIMIT_PROBLEMS.items():
        lib_, table, sd, S, ctrl, lin, con, sol, bound = joint_limit_problem(sched(), batch, seed)
        l_r, c_r = lin.copy(), con.copy()
        csd = sd.c()
        for b in range(batch):
            for i, ct in enumerate(ctrl):
                lb, cb = lin[b, i].copy(), con[b, i].copy()
                assert rl.ref_linearize_joint_limits(ctypes.byref(csd), ctypes.byref(table), ctypes.byref(ct), P(bound),
                                                     P(np.ascontiguousarray(sol[b, i])), P(lb), P(cb)) == 0
                l_r[b, i], c_r[b, i] = lb, cb
        data[f"jl_{which}_dlin"], data[f"jl_{which}_dcon"] = l_r - lin, c_r - con
    path = os.path.join(HERE, "golden_ref_stage_r2.npz")
    golden_io.save(path, data, record_sections(S, K, data), **PER_GRID_POINT)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")
    for which, seed in SEED_CASES.items():
        table, sd, S, K, ctrl, lin, con, sol, dx0 = seed_problem(which, seed, lib.orc_stage_layout_get, lib.orc_layout_get)
        out = ref_lib.reference_iteration(sd, S, K, table, ctrl, lin, con, dx0)
        data = {k: out[k] for k in SEED_KEYS}
        path = seed_path(which)
        golden_io.save(path, data, record_sections(S, K, data), **dict(PER_GRID_POINT, block=1 << 30))  # min_keep entries only
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")
