"""The reference's own outputs as the pin (tests/golden/golden_ref_r2.npz and golden_ref_seeds.npz, made by
tests/golden/make_golden_ref.py from the reference's src/riccati compiled unmodified):
  CPU:  the oracle (oracle/riccati_oracle.c) reproduces them -- this is what makes the oracle a trustworthy checker;
  CPU:  on further seeds, the oracle equals the reference on every field of every record;
  GPU:  the CUDA path reproduces them through the C ABI."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import golden_io  # noqa: E402
import make_golden_ref as mg  # noqa: E402

import oracle_lib  # noqa: E402
from robotoc_b200 import ANYMAL, Layout, ULayout  # noqa: E402

G = golden_io.load(os.path.join(HERE, "golden", "golden_ref_r2.npz"))
TOL = 1e-10  # relative to the array's scale; measured agreement oracle <-> reference code: 1e-15 .. 3e-15


def _rel(a, b):
    """Over the entries the fixture holds (golden_io)."""
    m = golden_io.finite(b)
    return float(np.max(np.abs(a[m] - b[m])) / max(np.max(np.abs(b[m])), 1e-300))


@pytest.mark.parametrize("name", list(mg.CASES))
def test_oracle_reproduces_reference_golden(name):
    lib = oracle_lib.load()
    L = Layout(ANYMAL, getter=lib.orc_layout_get)
    ctrl, kkt, dx0, full = mg.inputs(name, L)
    kk, ric, d, info = oracle_lib.riccati_batch(ANYMAL, L, ctrl, kkt, dx0)
    assert info == 0
    got = ric if full else mg.trim(L, ric)
    assert _rel(got, G[name + "_ric"]) < TOL
    assert _rel(d, G[name + "_dir"]) < TOL


def test_oracle_reproduces_reference_golden_unconstr():
    lib = oracle_lib.load()
    UL = ULayout(7, getter=lib.orc_ulayout_get)
    kkt, dx0 = mg.unconstr_inputs(UL)
    u = mg.UNCONSTR
    kk, ric, d, info = oracle_lib.unconstr_batch(7, UL, u["N"], u["dt"], kkt, dx0)
    assert info == 0
    assert _rel(ric, G["unconstr_ric"]) < TOL and _rel(d, G["unconstr_dir"]) < TOL


@pytest.fixture(scope="module")
def seeds():
    return golden_io.load(os.path.join(HERE, "golden", "golden_ref_seeds.npz"))


@pytest.mark.parametrize("name,seed", list(mg.FIELD_CASES.items()))
def test_oracle_equals_live_reference_every_field(seeds, name, seed):
    """Every field of every Riccati / direction record and the mutated KKT blocks (F, H, G, lu'), batch 3, fresh seeds."""
    lib = oracle_lib.load()
    L = Layout(ANYMAL, getter=lib.orc_layout_get)
    ctrl, kkt, dx0 = mg.field_inputs(name, seed, L)
    kk_o, ric_o, d_o, info = oracle_lib.riccati_batch(ANYMAL, L, ctrl, kkt, dx0)
    assert info == 0
    kk_r, ric_r, d_r = (seeds[f"field_{name}_{k}"] for k in ("kkt", "ric", "dir"))
    fields = sorted((getattr(L, f), f) for f in ("r_P r_s r_K r_k r_M r_m r_Psi r_Phi r_T r_W r_psix r_psiu r_phix r_phiu r_mt "
                                                  "r_mtn r_sc r_dtsdx r_stosc").split())
    ends = [o for o, _ in fields[1:]] + [L.r_stosc + 2]
    for (o, f), e in zip(fields, ends):
        a, b = ric_o[..., o:e], ric_r[..., o:e]
        m = golden_io.finite(b)
        assert m.all() or np.any(b[m]), f"{f}: the fixture holds none of the field's non-zeros"
        a, b = a[m], b[m]
        scale = np.max(np.abs(b))
        if scale == 0.0:
            assert np.max(np.abs(a)) == 0.0, f
        elif f == "r_W" and any(c.ns == ANYMAL.nu for c in ctrl):
            # ns == nu: W = -(Ginv - SDG^T DG) phi_u with an analytically zero matrix -> pure cancellation noise in both codes
            assert np.max(np.abs(a - b)) < 1e-9 * np.nanmax(np.abs(ric_r[..., L.r_T:L.r_T + ANYMAL.nu])), f
        else:
            assert np.max(np.abs(a - b)) < TOL * scale, f"{f}: {np.max(np.abs(a - b)) / scale:.2e}"
    assert _rel(d_o, d_r) < TOL
    assert _rel(kk_o, kk_r) < TOL  # in-place mutation semantics: Qxx, Qxu, Quu, lu <- F (- K^T G K), H, G, lu'


def test_oracle_equals_live_reference_unconstr(seeds):
    from synth import make_unconstr_kkt
    lib = oracle_lib.load()
    UL = ULayout(7, getter=lib.orc_ulayout_get)
    for N, dt, seed in mg.UNCONSTR_FIELD_CASES:
        kkt, dx0 = make_unconstr_kkt(7, UL, N, 3, seed)
        kk_o, ric_o, d_o, info = oracle_lib.unconstr_batch(7, UL, N, dt, kkt, dx0)
        kk_r, ric_r, d_r = (seeds[f"field_unconstr{N}_{k}"] for k in ("kkt", "ric", "dir"))
        assert info == 0 and _rel(ric_o, ric_r) < TOL and _rel(d_o, d_r) < TOL and _rel(kk_o, kk_r) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(mg.CASES))
def test_cuda_reproduces_reference_golden(name):
    from robotoc_b200 import RiccatiRecursion
    L = Layout(ANYMAL)
    ctrl, kkt, dx0, full = mg.inputs(name, L)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), kkt.shape[0])
    rr.setTimeDiscretization(ctrl)
    rr.backwardRiccatiRecursion(kkt)
    rr.forwardRiccatiRecursion(dx0)
    assert int(rr.info().max()) == 0
    ric, d = rr.getRiccatiFactorization(), rr.getDirection()
    ref_ric = G[name + "_ric"]
    if full:
        # stage-conditional sections the reference leaves at their constructor zeros are zero here too; W at ns == nu is noise
        got = ric
        for i, c in enumerate(ctrl):
            if c.ns == ANYMAL.nu:
                got[:, i, L.r_W:L.r_W + ANYMAL.nu] = ref_ric[:, i, L.r_W:L.r_W + ANYMAL.nu]
        assert _rel(got, ref_ric) < 1e-8
    else:
        assert _rel(mg.trim(L, ric), ref_ric) < 1e-8
    assert _rel(d, G[name + "_dir"]) < 1e-8
    rr.close()


@pytest.mark.gpu
def test_cuda_reproduces_reference_golden_unconstr():
    from robotoc_b200 import UnconstrRiccatiRecursion
    UL = ULayout(7)
    kkt, dx0 = mg.unconstr_inputs(UL)
    u = mg.UNCONSTR
    ur = UnconstrRiccatiRecursion(7, u["N"], u["dt"], u["batch"])
    ur.backwardRiccatiRecursion(kkt)
    ur.forwardRiccatiRecursion(dx0)
    assert int(ur.info().max()) == 0
    assert _rel(ur.getRiccatiFactorization(), G["unconstr_ric"]) < 1e-8
    assert _rel(ur.getDirection(), G["unconstr_dir"]) < 1e-8
    ur.close()
