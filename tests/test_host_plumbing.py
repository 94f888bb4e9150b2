"""The host layer of the constrained handle: bytes the host paths move over PCIe, kernel launches per call, and re-bound
device buffers.  The byte counts are computed here from the record layouts, independently of the library's own plan."""
import ctypes
import os

import numpy as np
import pytest

from helpers import crawl_schedule, jump_sto_schedule, small_event_schedule, trot_schedule
from robotoc_b200 import ANYMAL, DirectMultipleShooting, Layout, RiccatiRecursion, StageDims, StageLayout, anymal_constraint_table
from robotoc_b200.grid import IMPACT
from synth import make_stage_inputs, symmetrize_lin

pytestmark = pytest.mark.gpu

KKT, DX0, LIN, CON, SOL = 0, 4, 6, 7, 9
BATCH = 5
SCHEDULES = {
    "trot": lambda: trot_schedule(),
    "jump_sto": lambda: jump_sto_schedule(),
    "crawl_sto": lambda: crawl_schedule(sto=True),
    "small_event": lambda: small_event_schedule(),
}


def _setup(ctrl, batch=BATCH):
    table = anymal_constraint_table()
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    rr = RiccatiRecursion(ANYMAL, len(ctrl), batch)
    rr.setTimeDiscretization(ctrl)
    return rr, DirectMultipleShooting(rr, sd, table), sd, StageLayout(sd), Layout(ANYMAL)


def _expected_bytes(rr, sd, S, K, ctrl):
    """(upload bytes per buffer, {mode: (h2d, d2h)}) from the layouts: what the kernels read or what persists, nothing else."""
    G, B = len(ctrl), rr.batch
    n_sw = sum(1 for c in ctrl if c.ns > 0 and c.type != IMPACT)  # stages whose linearization carries a switching section
    n_extra = sum(1 for c in ctrl if c.ns > 0 or c.sto)          # stages whose KKT record carries extras
    sw = n_sw * (S.l_ha - S.l_Phix)
    lin = G * (S.l_Phix + S.l_dgdf + ((15 * S.ncon + 1) & ~1) - S.l_ha) + sw
    if 2 * n_extra > G:
        kkt = G * (K.k_core_size + K.k_extra_size)
    else:
        kkt = G * K.k_core_size + n_extra * K.k_extra_size
    wire = int(rr._lib.rbt_wire_doubles(ctypes.byref(sd.c()), ctrl, G, 0))
    con_in, sol, dx0 = G * 3 * S.ncp, G * S.s_stride, K.nx
    down = G * S.s_stride + G * 2 * S.ncp + 2  # solution, slack | dual, step sizes
    upload = {KKT: kkt, LIN: lin, CON: con_in, SOL: sol, DX0: dx0}
    modes = {"dense": (lin + con_in + sol + dx0, down), "wire": (wire + sw + con_in + sol + dx0, down),
             "resident": (wire + sw + G * S.ncp + dx0, down)}
    return ({k: 8 * B * v for k, v in upload.items()},
            {m: (8 * B * u, 8 * B * d) for m, (u, d) in modes.items()})


@pytest.mark.parametrize("name", list(SCHEDULES))
def test_cuda_transfer_bytes_match_the_record_layouts(name):
    _, _, ctrl = SCHEDULES[name]()
    rr, dms, sd, S, K = _setup(ctrl)
    try:
        upload, modes = _expected_bytes(rr, sd, S, K, ctrl)
        for which, n in upload.items():
            assert int(rr._lib.rbt_upload_bytes(rr._h, which)) == n, which
        assert dms.iteration_host_bytes() == modes["dense"]
        assert dms.iteration_host_bytes(wire=True) == modes["wire"]
        assert dms.iteration_host_bytes(resident=True) == modes["resident"]
    finally:
        rr.close()


def _inputs(sd, S, ctrl):
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, BATCH, 3)
    return symmetrize_lin(S, lin), con, sol, dx0


def _step_by_step(rr, dms, lin, con, sol, dx0):
    dms.setSolution(sol)
    dms.condense(lin, con)
    rr.backwardRiccatiRecursion()
    rr.forwardRiccatiRecursion(dx0)
    dms.computeStepSizes()
    dms.integrateSolution()
    rr.synchronize()


def test_cuda_launch_counts():
    _, _, ctrl = small_event_schedule()
    rr, dms, sd, S, K = _setup(ctrl)
    try:
        lin, con, sol, dx0 = _inputs(sd, S, ctrl)
        n0 = rr.launch_count()
        _step_by_step(rr, dms, lin, con, sol, dx0)
        assert rr.launch_count() - n0 == 6  # mjtjinv + condense, backward (structure known), forward, expand, update
        kkt = dms.getKKT()
        n0 = rr.launch_count()
        rr.backwardRiccatiRecursion(kkt)  # uploaded records under RBT_FXX_AUTO: structure check + both instances
        rr.synchronize()
        assert rr.launch_count() - n0 == 3
        res = np.ascontiguousarray(con[:, :, S.c_res:S.c_res + S.ncp])
        runs = {"dense": (lambda: dms.iteration_host(lin, con, sol, dx0), 6),
                "wire": (lambda: dms.iteration_host_wire(dms.pack_wire(lin), lin, con, sol, dx0), 7),  # + unpack_wire
                "resident": (lambda: dms.iteration_host_resident(dms.pack_wire(lin), lin, res, dx0), 8)}  # + pack_slack_dual
        for chunks in (1, 3):
            os.environ["RBT_E2E_CHUNKS"] = str(chunks)
            try:
                for mode, (run, per_chunk) in runs.items():
                    n0 = rr.launch_count()
                    run()
                    assert rr.launch_count() - n0 == per_chunk * chunks, (mode, chunks)
            finally:
                del os.environ["RBT_E2E_CHUNKS"]
    finally:
        rr.close()


def test_cuda_bind_buffer_round_trip():
    torch = pytest.importorskip("torch")
    _, _, ctrl = small_event_schedule()
    rr, dms, sd, S, K = _setup(ctrl)
    try:
        lin, con, sol, dx0 = _inputs(sd, S, ctrl)
        own = rr.dev_ptr(SOL)
        t = torch.zeros(rr.buf_doubles(SOL), dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()
        rr.bind_buffer(SOL, ctypes.c_void_p(t.data_ptr()))
        assert rr.dev_ptr(SOL) == t.data_ptr()
        _step_by_step(rr, dms, lin, con, sol, dx0)
        bound = dms.getSolution()
        rr.bind_buffer(SOL, None)
        assert rr.dev_ptr(SOL) == own
        _step_by_step(rr, dms, lin, con, sol, dx0)  # same inputs, now into the handle's own buffer
        np.testing.assert_array_equal(dms.getSolution(), bound)
        rr.close()
        got = t.cpu().numpy().reshape(bound.shape)  # the caller's buffer outlives the handle, holding the bound run's result
        np.testing.assert_array_equal(got, bound)
        assert not np.array_equal(bound, sol)
    finally:
        rr.close()  # idempotent
