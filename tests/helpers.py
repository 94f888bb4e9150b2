"""Shared test helpers: problems, record views, dense KKT reference solve."""
import numpy as np

from robotoc_b200 import ANYMAL, Layout
from robotoc_b200.grid import IMPACT, LIFT, TERMINAL
from schedule_fixture import (ContactEvents, TimeDiscretization, stage_ctrl_array, anymal_crawl_events, anymal_trot_events,
                              anymal_jump_sto_events)
from synth import make_kkt, mat


def small_event_schedule(sto=False):
    """ANYmal, T=0.4, N=8: lift at 0.07, impact (dimf 6) at 0.23 -> Lift, Impact, one switching-constraint stage."""
    ev = ContactEvents(phase_dimf=[12], phase_mask=[0b1111])
    ev.push_back(False, 0.07, 6, sto=sto, post_mask=0b1001)
    ev.push_back(True, 0.23, 12, impact_dimf=6, sto=sto, post_mask=0b1111, impact_mask=0b0110)
    td = TimeDiscretization(0.4, 8).discretize(ev, 0.0, sto=sto)
    return td, ev, stage_ctrl_array(td, ev)


def trot_schedule(N=40):
    ev = anymal_trot_events()
    td = TimeDiscretization(1.12, N).discretize(ev, 0.0)
    return td, ev, stage_ctrl_array(td, ev)


def jump_sto_schedule(N=80):
    ev = anymal_jump_sto_events()
    td = TimeDiscretization(1.7, N).discretize(ev, 0.0, sto=True)
    return td, ev, stage_ctrl_array(td, ev)


CRAWL_SIZES = {"crawl_full": dict(cycle=2, swing=0.5, ds=0.04),   # examples/anymal/crawl.cpp itself: N = 210, 219 grid points
               "crawl_small": dict(cycle=1, swing=0.1, ds=0.04)}  # every event kind and contact dimension: N = 26, 31 grid points


def crawl_schedule(size="crawl_small", sto=False, dt=0.02):
    """ANYmal crawl (schedule_fixture.anymal_crawl_events): phases with three feet in contact (nf = 9), single-foot impacts
    (nf = 3 on the Impact stage, ns = 3 on the switching-constraint stage before it).  N = T / dt as crawl.cpp computes it."""
    p = CRAWL_SIZES[size]
    ev = anymal_crawl_events(p["cycle"], p["swing"], p["ds"], sto=sto)
    T = p["ds"] + p["cycle"] * (4 * p["swing"] + 2 * p["ds"])
    td = TimeDiscretization(T, int(T / dt)).discretize(ev, 0.0, sto=sto)
    return td, ev, stage_ctrl_array(td, ev)


def dense_kkt_solve(dims, L, ctrl, kkt1, dx0):
    """Independent reference: assemble the full block KKT system of the equality-constrained LQ subproblem
    (no STO) for ONE OCP and solve it with numpy.  Returns dict of per-stage dx, du, lmd, xi."""
    n_grid = len(ctrl)
    N = n_grid - 1
    nx, nu, nv = dims.nx, dims.nu, dims.nv
    idx = {}
    n = 0

    def alloc(name, i, size):
        nonlocal n
        idx[(name, i)] = slice(n, n + size)
        n += size

    for i in range(n_grid):
        alloc("dx", i, nx)
        alloc("lmd", i, nx)
        if i < N and ctrl[i].type != IMPACT:
            alloc("du", i, nu)
            if ctrl[i].ns > 0:
                alloc("xi", i, ctrl[i].ns)
    Kmat = np.zeros((n, n))
    rhs = np.zeros(n)
    I = np.eye(nx)
    # row blocks are indexed by the variable whose stationarity / constraint they express
    for i in range(n_grid):
        rec = kkt1[i]
        sx, sl = idx[("dx", i)], idx[("lmd", i)]
        Qxx = mat(rec, L.k_Qxx, nx, nx)
        lx = rec[L.k_lx:L.k_lx + nx]
        # stationarity wrt dx_i : Qxx dx + Qxu du + lx + A^T lmd_{i+1} - lmd_i + C^T xi = 0
        Kmat[sx, sx] += Qxx
        Kmat[sx, sl] += -I
        rhs[sx] += -lx
        # constraint paired with lmd_i : (i=0) dx_0 = dx0 ; (i>0) A dx_{i-1} + B du_{i-1} + Fx - dx_i = 0
        if i == 0:
            Kmat[sl, sx] += I
            rhs[sl] += dx0
        if i < N:
            A = mat(rec, L.k_Fxx, nx, nx)
            Fx = rec[L.k_Fx:L.k_Fx + nx]
            sxn, sln = idx[("dx", i + 1)], idx[("lmd", i + 1)]
            Kmat[sx, sln] += A.T
            Kmat[sln, sx] += A
            Kmat[sln, sxn] += -I
            rhs[sln] += -Fx
            if ctrl[i].type != IMPACT:
                su = idx[("du", i)]
                Qxu = mat(rec, L.k_Qxu, nx, nu)
                Quu = mat(rec, L.k_Quu, nu, nu)
                lu = rec[L.k_lu:L.k_lu + nu]
                B = np.zeros((nx, nu))
                B[nv:, :] = mat(rec, L.k_Fvu, nv, nu)
                Kmat[sx, su] += Qxu
                Kmat[su, sx] += Qxu.T
                Kmat[su, su] += Quu
                Kmat[su, sln] += B.T
                Kmat[sln, su] += B
                rhs[su] += -lu
                ns = ctrl[i].ns
                if ns > 0:
                    sxi = idx[("xi", i)]
                    C = mat(rec, L.k_Phix, ns, nx)
                    D = mat(rec, L.k_Phiu, ns, nu)
                    p = rec[L.k_p:L.k_p + ns]
                    Kmat[sx, sxi] += C.T
                    Kmat[su, sxi] += D.T
                    Kmat[sxi, sx] += C
                    Kmat[sxi, su] += D
                    rhs[sxi] += -p
    sol = np.linalg.solve(Kmat, rhs)
    return {k: sol[v] for k, v in idx.items()}


def dense_kkt_solve_sto(dims, L, ctrl, kkt1, dx0):
    """Independent reference for the switching-time-optimisation path: the full KKT system of the LQ sub-problem with
    the switching-time increments ts_k of all events as unknowns (every event STO-enabled), ONE OCP, numpy dense solve.
    A stage of the phase between events p and p+1 sees Delta = ts_{p+1} - ts_p through fx (dynamics), hx / hu / h (cost
    gradient), Phit (switching constraint) and the quadratic 0.5*Qtt*Delta^2 - Qtt_prev*Delta*ts_{p+1}; the last form is
    what the reference's accumulation xi += Qtt, chi += Qtt_prev (backward_riccati_recursion_factorizer.cpp:108-120)
    amounts to in the value function 0.5*xi*Delta^2 - chi*Delta*b + 0.5*rho*b^2 that its phase transition
    (riccati_factorizer.cpp:145-175) minimises.  Returns (solution dict, phase of every grid, number of events)."""
    n_grid = len(ctrl); N = n_grid - 1
    nx, nu, nv = dims.nx, dims.nu, dims.nv
    # phase of every grid; events are numbered 1..E; phase p lies between event p and event p+1
    phase = []; p = 0
    for i in range(n_grid):
        if ctrl[i].type == LIFT: p += 1
        phase.append(p)
        if ctrl[i].type == IMPACT: p += 1
    E = p
    idx = {}; n = 0
    def alloc(name, i, size):
        nonlocal n
        idx[(name, i)] = slice(n, n + size); n += size
    for i in range(n_grid):
        alloc("dx", i, nx); alloc("lmd", i, nx)
        if i < N and ctrl[i].type != IMPACT:
            alloc("du", i, nu)
            if ctrl[i].ns > 0: alloc("xi", i, ctrl[i].ns)
    for k in range(1, E + 1): alloc("ts", k, 1)
    K = np.zeros((n, n)); rhs = np.zeros(n); I = np.eye(nx)
    def ts_terms(p):
        out = []
        if p + 1 <= E: out.append((idx[("ts", p + 1)], +1.0))
        if p >= 1: out.append((idx[("ts", p)], -1.0))
        return out
    for i in range(n_grid):
        rec = kkt1[i]; sx, sl = idx[("dx", i)], idx[("lmd", i)]
        K[sx, sx] += mat(rec, L.k_Qxx, nx, nx); K[sx, sl] += -I; rhs[sx] += -rec[L.k_lx:L.k_lx + nx]
        if i == 0:
            K[sl, sx] += I; rhs[sl] += dx0
        if i < N:
            A = mat(rec, L.k_Fxx, nx, nx); Fx = rec[L.k_Fx:L.k_Fx + nx]
            sxn, sln = idx[("dx", i + 1)], idx[("lmd", i + 1)]
            K[sx, sln] += A.T; K[sln, sx] += A; K[sln, sxn] += -I; rhs[sln] += -Fx
            if ctrl[i].type != IMPACT:
                su = idx[("du", i)]
                Qxu = mat(rec, L.k_Qxu, nx, nu); Quu = mat(rec, L.k_Quu, nu, nu)
                B = np.zeros((nx, nu)); B[nv:, :] = mat(rec, L.k_Fvu, nv, nu)
                K[sx, su] += Qxu; K[su, sx] += Qxu.T; K[su, su] += Quu; K[su, sln] += B.T; K[sln, su] += B
                rhs[su] += -rec[L.k_lu:L.k_lu + nu]
                ns = ctrl[i].ns
                if ns > 0:
                    sxi = idx[("xi", i)]
                    C = mat(rec, L.k_Phix, ns, nx); D = mat(rec, L.k_Phiu, ns, nu)
                    K[sx, sxi] += C.T; K[su, sxi] += D.T; K[sxi, sx] += C; K[sxi, su] += D; rhs[sxi] += -rec[L.k_p:L.k_p + ns]
                if ctrl[i].sto:
                    fx = rec[L.k_fx:L.k_fx + nx]; hx = rec[L.k_hx:L.k_hx + nx]; hu = rec[L.k_hu:L.k_hu + nu]
                    Qtt, h = rec[L.k_sc + 0], rec[L.k_sc + 2]
                    tt = ts_terms(phase[i])
                    for (st, sg) in tt:
                        K[sx, st] += sg * hx[:, None]; K[st, sx] += sg * hx[None, :]
                        K[su, st] += sg * hu[:, None]; K[st, su] += sg * hu[None, :]
                        K[sln, st] += sg * fx[:, None]; K[st, sln] += sg * fx[None, :]
                        rhs[st] += -sg * h
                        if ns > 0:
                            Pt = rec[L.k_Phit:L.k_Phit + ns]
                            K[sxi, st] += sg * Pt[:, None]; K[st, sxi] += sg * Pt[None, :]
                        for (st2, sg2) in tt:
                            K[st, st2] += sg * sg2 * Qtt
                    # recursion-implied cross term: - Qtt_prev * (b - a) * b
                    Qtp = rec[L.k_sc + 1]
                    pp = phase[i]
                    if pp + 1 <= E:
                        sb = idx[("ts", pp + 1)]
                        K[sb, sb] += -2.0 * Qtp
                        if pp >= 1:
                            sa = idx[("ts", pp)]
                            K[sa, sb] += Qtp; K[sb, sa] += Qtp
    sol = np.linalg.solve(K, rhs)
    return {k: sol[v] for k, v in idx.items()}, phase, E


def rel_err(a, b):
    """max |a-b| / max(|b|, tiny) over the array (relative to the block's scale, like Eigen isApprox)."""
    a, b = np.asarray(a), np.asarray(b)
    denom = max(np.max(np.abs(b)), 1e-300)
    return float(np.max(np.abs(a - b)) / denom)
