"""Generates tests/golden/golden_ref_r2.npz from the REFERENCE's own code: oracle/_ref/libref_riccati.so is the reference's
src/riccati/*.cpp + src/core/split_*.cpp compiled unmodified (oracle/Makefile.ref, Eigen / Robot stand-ins of oracle/shim).
Only runs where a checkout of the reference is available (ROBOTOC_REFERENCE, see oracle/Makefile.ref):

    python tests/golden/make_golden_ref.py

Inputs are regenerated from the seeds below by the tests (tests/synth.py); only the reference's outputs are stored, sampled
by golden_io.  golden_ref_r2.npz:
  - full Riccati + direction records for the small event schedules (with / without switching-time optimisation) and the
    iiwa14 recursion, and [P|s|K|k], the STO scalars / policies and the direction records for the BASELINE schedules (trot
    N=40, jump STO N=80).
golden_ref_seeds.npz:
  - "field_*": every Riccati / direction record and the KKT blocks the recursion mutates, batch 3, on further seeds
    (FIELD_CASES, UNCONSTR_FIELD_CASES);
  - "filter_*": accepted step size and trial index of the reference's LineSearchFilter over consecutive line searches
    (filter_cases()).
tests/test_golden_ref.py and tests/test_line_search.py check the oracle (CPU) and the CUDA path (-m gpu) against these files.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import jump_sto_schedule, small_event_schedule, trot_schedule  # noqa: E402
from robotoc_b200 import ANYMAL  # noqa: E402
from synth import make_kkt, make_unconstr_kkt  # noqa: E402

import golden_io  # noqa: E402

CASES = {  # name -> (schedule factory, seed, batch, store full records?)
    "small": (lambda: small_event_schedule(False), 201, 1, True),
    "small_sto": (lambda: small_event_schedule(True), 202, 1, True),
    "trot_n40": (lambda: trot_schedule(40), 203, 1, False),
    "jump_sto_n80": (lambda: jump_sto_schedule(80), 204, 1, False),
}
UNCONSTR = dict(nv=7, N=20, dt=0.05, seed=205, batch=2)
FIELD_CASES = {"small": 31, "small_sto": 32, "trot_n40": 33, "jump_sto_n80": 34}  # name -> seed, batch 3
UNCONSTR_FIELD_CASES = ((20, 0.05, 41), (50, 0.02, 42))                           # (N, dt, seed), batch 3
FILTER = dict(cases=20, rounds=40, n_trials=8, rate=0.75, min_step=0.05, cost_reduction=0.005, violation_reduction=0.005)


def inputs(name, L):
    sched, seed, batch, full = CASES[name]
    td, ev, ctrl = sched()
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=batch, seed=seed)
    return ctrl, kkt, dx0, full


def trim(L, ric):
    """[P|s|K|k] + {xi, chi, rho, eta, iota} + STOPolicy of every stage."""
    return np.concatenate([ric[..., :L.r_core_size], ric[..., L.r_sc:L.r_sc + 5], ric[..., L.r_dtsdx:L.r_stosc + 2]], axis=-1)


def trim_sections(L):
    """golden_io section offsets of a trim()med record."""
    sc = L.r_core_size
    return [L.r_P, L.r_s, L.r_K, L.r_k, sc, sc + 5, sc + 5 + L.r_stosc - L.r_dtsdx]


def record_sections(L, UL, keys):
    """golden_io section offsets of the records this file stores, by key."""
    out = {}
    for key in keys:
        layout = UL if "unconstr" in key else L
        if key.endswith("_ric"):
            trimmed = key[:-4] in CASES and not CASES[key[:-4]][3]
            out[key] = trim_sections(L) if trimmed else golden_io.sections(layout, "r_")
        elif key.endswith("_dir"):
            out[key] = golden_io.sections(layout, "d_")
        elif key.endswith("_kkt"):
            out[key] = golden_io.sections(layout, "k_")
    return out


def unconstr_inputs(UL):
    u = UNCONSTR
    return make_unconstr_kkt(u["nv"], UL, u["N"], u["batch"], u["seed"])


def field_inputs(name, seed, L):
    td, ev, ctrl = CASES[name][0]()
    kkt, dx0 = make_kkt(ANYMAL, L, ctrl, batch=3, seed=seed)
    return ctrl, kkt, dx0


def filter_cases():
    """Per case: (alpha_max, cost0, violation0, cost, violation) of FILTER["rounds"] consecutive line searches whose costs drift
    down like a converging solver's and whose violations shrink."""
    rng = np.random.default_rng(3)
    rounds, n_trials = FILTER["rounds"], FILTER["n_trials"]
    for case in range(FILTER["cases"]):
        amax = rng.uniform(0.05, 1.0, size=rounds)
        trend = np.linspace(10.0, 1.0, rounds)[:, None]
        cost = trend + rng.normal(0, 0.5, size=(rounds, n_trials))
        viol = np.abs(trend * 0.1 + rng.normal(0, 0.05, size=(rounds, n_trials)))
        yield amax, cost[:, 0] + 0.1, viol[:, 0] + 0.01, cost, viol


if __name__ == "__main__":
    import ctypes

    import oracle_lib
    import ref_lib
    from robotoc_b200 import Layout, ULayout
    lib = oracle_lib.load()
    L = Layout(ANYMAL, getter=lib.orc_layout_get)
    out = {}
    for name in CASES:
        ctrl, kkt, dx0, full = inputs(name, L)
        kk, ric, d = ref_lib.riccati_batch(ANYMAL, L, ctrl, kkt, dx0)
        out[name + "_ric"] = ric if full else trim(L, ric)
        out[name + "_dir"] = d
    UL = ULayout(7, getter=lib.orc_ulayout_get)
    kkt, dx0 = unconstr_inputs(UL)
    kk, ric, d = ref_lib.unconstr_batch(7, UL, UNCONSTR["N"], UNCONSTR["dt"], kkt, dx0)
    out["unconstr_ric"], out["unconstr_dir"] = ric, d
    path = os.path.join(HERE, "golden_ref_r2.npz")
    golden_io.save(path, out, record_sections(L, UL, out))
    out = {}
    for name, seed in FIELD_CASES.items():
        ctrl, kkt, dx0 = field_inputs(name, seed, L)
        out[f"field_{name}_kkt"], out[f"field_{name}_ric"], out[f"field_{name}_dir"] = ref_lib.riccati_batch(ANYMAL, L, ctrl, kkt, dx0)
    for N, dt, seed in UNCONSTR_FIELD_CASES:
        kkt, dx0 = make_unconstr_kkt(7, UL, N, 3, seed)
        out[f"field_unconstr{N}_kkt"], out[f"field_unconstr{N}_ric"], out[f"field_unconstr{N}_dir"] = ref_lib.unconstr_batch(7, UL, N, dt, kkt, dx0)
    ref = ref_lib.load()
    ref.ref_filter_line_search.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_double] * 4 + [ctypes.c_void_p] * 7
    f, P = FILTER, oracle_lib.ptr
    steps, ks = np.zeros((f["cases"], f["rounds"])), np.zeros((f["cases"], f["rounds"]))
    for case, (amax, cost0, viol0, cost, viol) in enumerate(filter_cases()):
        k = np.zeros(f["rounds"], dtype=np.int32)
        ref.ref_filter_line_search(f["rounds"], f["n_trials"], f["rate"], f["min_step"], f["cost_reduction"], f["violation_reduction"],
                                   P(amax), P(cost0), P(viol0), P(np.ascontiguousarray(cost)), P(np.ascontiguousarray(viol)),
                                   P(steps[case]), k.ctypes.data_as(ctypes.c_void_p))
        ks[case] = k
    out["filter_step"], out["filter_k"] = steps, ks
    path_seeds = os.path.join(HERE, "golden_ref_seeds.npz")
    golden_io.save(path_seeds, out, record_sections(L, UL, out), block=64)  # batch 3 on long horizons: a thinner sample
    print("wrote", path, os.path.getsize(path) // 1024, "KiB,", path_seeds, os.path.getsize(path_seeds) // 1024, "KiB;",
          ref.ref_version().decode())
