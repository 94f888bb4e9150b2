"""TEST FIXTURE (not product code): control-table producer for the BASELINE schedules.

Restates robotoc::TimeDiscretization::discretize / correctTimeSteps
(/root/reference/src/ocp/time_discretization.cpp:43-262) and the event bookkeeping of
robotoc::ContactSequence (/root/reference/src/planner/contact_sequence.cpp:55-95) as far as the
kernels need it: the per-grid-point GridInfo (grid_info.hpp:25-92) and, from it, the rbt_stage_ctrl
table shared by a batch of OCPs.  A real drop-in takes GridInfo from robotoc's own class.
"""
import math
from dataclasses import dataclass, field
from typing import List

from robotoc_b200 import _lib
from robotoc_b200.grid import GridInfo, INTERMEDIATE, IMPACT, LIFT, TERMINAL, plain_schedule  # noqa: F401

_EPS = math.sqrt(2.220446049250313e-16)


@dataclass
class ContactEvents:
    """The part of ContactSequence the discretization reads: event times, kinds, STO flags and the
    contact dimension of every phase (dimf) / every impact (impact dimf)."""
    impact_times: List[float] = field(default_factory=list)
    lift_times: List[float] = field(default_factory=list)
    sto_impact: List[bool] = field(default_factory=list)
    sto_lift: List[bool] = field(default_factory=list)
    phase_dimf: List[int] = field(default_factory=lambda: [0])   # dimf of contactStatus(phase)
    impact_dimf: List[int] = field(default_factory=list)         # dimf of impactStatus(impact_index)
    phase_mask: List[int] = field(default_factory=lambda: [0])   # active point contacts of contactStatus(phase), bit per contact
    impact_mask: List[int] = field(default_factory=list)         # contacts of impactStatus(impact_index)

    def push_back(self, is_impact: bool, time: float, post_dimf: int, impact_dimf: int = 0, sto: bool = False,
                  post_mask: int = None, impact_mask: int = 0):
        """ContactSequence::push_back (contact_sequence.cpp:55-95): an event is an Impact iff new contacts close."""
        if is_impact:
            self.impact_times.append(time)
            self.sto_impact.append(sto)
            self.impact_dimf.append(impact_dimf)
            if 3 * bin(impact_mask).count("1") != impact_dimf:
                raise ValueError("[ContactEvents] impact_mask must name exactly impact_dimf / 3 contacts")
            self.impact_mask.append(impact_mask)
        else:
            self.lift_times.append(time)
            self.sto_lift.append(sto)
        self.phase_dimf.append(post_dimf)
        if post_mask is None or 3 * bin(post_mask).count("1") != post_dimf:
            raise ValueError("[ContactEvents] post_mask must be given and name exactly post_dimf / 3 contacts")
        self.phase_mask.append(post_mask)


class TimeDiscretization:
    """TimeDiscretization(T, N, reserved_num_discrete_events) -- time_discretization.cpp:9-27."""

    def __init__(self, T: float, N: int):
        if T <= 0:
            raise ValueError("[TimeDiscretization] invalid argument: 'T' must be positive!")
        if N <= 0:
            raise ValueError("[TimeDiscretization] invalid argument: 'N' must be positive!")
        self.T, self.N = T, N
        self.grid: List[GridInfo] = []
        self.num_grids = 0

    def size(self):
        return self.num_grids + 1

    def __len__(self):
        return self.size()

    def __getitem__(self, i):
        return self.grid[i]

    def discretize(self, ev: ContactEvents, t: float = 0.0, sto: bool = True):
        """discretize (time_discretization.cpp:43-183); with sto=True followed by correctTimeSteps (:186-262): the
        per-phase uniform time steps and the STO flags, as OCPSolver applies it to PhaseBased / STO problems."""
        T, N_ = self.T, self.N
        n_imp, n_lift = len(ev.impact_times), len(ev.lift_times)
        size = N_ + n_lift + 2 * n_imp + 1
        g = [GridInfo() for _ in range(size + 1)]
        ni = 0
        nl = 0
        while ni < n_imp and not ev.impact_times[ni] > t:
            ni += 1
        while nl < n_lift and not ev.lift_times[nl] > t:
            nl += 1
        dt = T / N_
        margin = 0.5 * dt
        stage = 0
        ti = t

        def fill(st, tt, dtt, typ):
            g[st].t, g[st].dt, g[st].stage = tt, dtt, st
            g[st].phase = ni + nl
            g[st].impact_index = ni - 1
            g[st].lift_index = nl - 1
            g[st].type = typ

        while ti + _EPS < t + T:
            has_imp = ni < n_imp
            has_lift = nl < n_lift
            fill(stage, ti, dt, INTERMEDIATE)
            if has_imp:
                nt = ev.impact_times[ni]
                if nt <= ti + dt + _EPS and (nt + margin < t + T):
                    g[stage].dt = nt - ti
                    stage += 1
                    ni += 1
                    fill(stage, nt, 0.0, IMPACT)
                    stage += 1
                    fill(stage, nt, min(ti + dt, t + T) - nt, INTERMEDIATE)
                    if abs((ti + dt) - nt) < _EPS:
                        ti += dt
                        g[stage].dt = ti + dt - nt
            if has_lift:
                nt = ev.lift_times[nl]
                if nt <= ti + dt + _EPS and (nt + margin < t + T):
                    g[stage].dt = nt - ti
                    stage += 1
                    nl += 1
                    fill(stage, nt, min(ti + dt, t + T) - nt, LIFT)
                    if abs((ti + dt) - nt) < _EPS:
                        ti += dt
                        g[stage].dt = ti + dt - nt
            stage += 1
            ti += dt
        fill(stage, t + T, 0.0, TERMINAL)
        ng = stage
        for i in range(ng):
            g[i].dt_next = g[i + 1].dt
        g[ng].dt_next = 0.0
        for i in range(ng - 1):
            g[i].switching_constraint = (g[i + 2].type == IMPACT)
        g[ng - 1].switching_constraint = False
        g[ng].switching_constraint = False
        for i in range(ng + 1):
            g[i].t0 = t
            g[i].sto = False
            g[i].sto_next = False
            g[i].stage_in_phase = 1
            g[i].num_grids_in_phase = 1
        # count grids (:148-182)
        sip = 0
        pstart = 0
        i = 0
        while i < ng:
            if g[i].type == IMPACT:
                for j in range(pstart, i):
                    g[j].num_grids_in_phase = sip
                g[i].stage_in_phase = 0
                g[i].num_grids_in_phase = 0
                i += 1
                sip = 0
                pstart = i
            elif g[i].type == LIFT:
                for j in range(pstart, i):
                    g[j].num_grids_in_phase = sip
                sip = 0
                pstart = i
            g[i].stage_in_phase = sip
            sip += 1
            i += 1
        for j in range(pstart, ng):
            g[j].num_grids_in_phase = sip
        g[ng].stage_in_phase = 0
        g[ng].num_grids_in_phase = 0
        self.grid = g[:ng + 1]
        self.num_grids = ng
        if sto:
            self._correct_time_steps(ev, t)
            self._set_sto(ev)
        return self

    def _correct_time_steps(self, ev: ContactEvents, t: float):
        """Per-phase uniform dt / t: time_discretization.cpp:186-225."""
        g, ng = self.grid, self.num_grids
        prev_stage, prev_time = 0, t
        i = 0
        while i < ng:
            if g[i].type == IMPACT:
                et = ev.impact_times[g[i + 1].impact_index]
                dt = (et - prev_time) / g[i - 1].num_grids_in_phase
                for j in range(prev_stage, i):
                    g[j].t = prev_time + (j - prev_stage) * dt
                    g[j].dt = dt
                g[i].t, g[i].dt = et, 0.0
                prev_time, prev_stage = et, i + 1
                i += 1
            elif g[i + 1].type == LIFT:
                et = ev.lift_times[g[i + 1].lift_index]
                dt = (et - prev_time) / g[i].num_grids_in_phase
                for j in range(prev_stage, i + 1):
                    g[j].t = prev_time + (j - prev_stage) * dt
                    g[j].dt = dt
                prev_time, prev_stage = et, i + 1
            elif g[i + 1].type == TERMINAL:
                dt = (t + self.T - prev_time) / g[i].num_grids_in_phase
                for j in range(prev_stage, i + 1):
                    g[j].t = prev_time + (j - prev_stage) * dt
                    g[j].dt = dt
            i += 1
        g[ng].t, g[ng].dt = t + self.T, 0.0
        for i in range(ng):
            g[i].dt_next = g[i + 1].dt
        g[ng].dt_next = 0.0

    def _set_sto(self, ev: ContactEvents):
        """STO flags: time_discretization.cpp:228-261."""
        g, ng = self.grid, self.num_grids
        sto_event = []
        for i in range(ng):
            if g[i].type == IMPACT:
                sto_event.append(bool(ev.sto_impact[g[i + 1].impact_index]))
            elif g[i].type == LIFT:
                sto_event.append(bool(ev.sto_lift[g[i + 1].lift_index]))
        if not sto_event:
            return
        sto_phase = [sto_event[0]]
        for i in range(1, len(sto_event)):
            sto_phase.append(sto_event[i - 1] or sto_event[i])
        sto_phase.append(sto_event[-1])
        sto_phase.append(False)
        for i in range(ng):
            ph = g[i].phase - g[0].phase
            g[i].sto = sto_phase[ph]
            g[i].sto_next = sto_phase[ph + 1]
        g[ng].sto = False
        g[ng].sto_next = False


def stage_ctrl_array(td: TimeDiscretization, ev: ContactEvents):
    """GridInfo list -> ctypes array of rbt_stage_ctrl.  The switching-constraint dimension of grid i is the
    impact dimf of impactStatus(impact_index+1) (ocp_solver.cpp:471-474, kkt_factory.cpp:75-79)."""
    n = td.size()
    arr = (_lib.rbt_stage_ctrl * n)()
    for i, gi in enumerate(td.grid):
        c = arr[i]
        c.type = gi.type
        c.sto = int(gi.sto)
        c.sto_next = int(gi.sto_next)
        c.ns = ev.impact_dimf[gi.impact_index + 1] if gi.switching_constraint else 0
        if gi.type == IMPACT:
            c.nf = ev.impact_dimf[gi.impact_index]
            c.contact_mask = ev.impact_mask[gi.impact_index]
        else:
            c.nf = ev.phase_dimf[gi.phase] if gi.phase < len(ev.phase_dimf) else 0
            c.contact_mask = ev.phase_mask[gi.phase] if gi.phase < len(ev.phase_mask) else 0
        c.ngrids_in_phase = gi.num_grids_in_phase
        c.dt = gi.dt
        c.ineq_gate = max(0, 2 - gi.stage) if gi.type in (INTERMEDIATE, LIFT) else 0  # ConstraintsData::setTimeStage(grid.stage)
    return arr


def anymal_trot_events() -> ContactEvents:
    """Contact schedule of /root/reference/examples/anymal/trot.cpp:41-47,172-190 (cycle=1):
    stand(12) -lift@0.04-> LF+RH(6) -impact@0.54-> stand -lift@0.58-> LH+RF(6) -impact@1.08-> stand; T=1.12."""
    # contact order LF, LH, RF, RH (trot.cpp:34-37)
    ev = ContactEvents(phase_dimf=[12], phase_mask=[0b1111])
    t0, swing, ds = 0.04, 0.5, 0.04
    ev.push_back(False, t0, 6, post_mask=0b1001)                                       # LH, RF swing
    ev.push_back(True, t0 + swing, 12, impact_dimf=6, post_mask=0b1111, impact_mask=0b0110)
    ev.push_back(False, t0 + swing + ds, 6, post_mask=0b0110)                          # LF, RH swing
    ev.push_back(True, t0 + 2 * swing + ds, 12, impact_dimf=6, post_mask=0b1111, impact_mask=0b1001)
    return ev


def anymal_crawl_events(cycle: int = 2, swing: float = 0.5, ds: float = 0.04, sto: bool = False) -> ContactEvents:
    """Contact schedule of /root/reference/examples/anymal/crawl.cpp:43-46,161-229: one foot in the air at a time, per cycle
    stand(12) -lift RH-> (9) -RH closes, RF opens-> (9) -RF closes-> stand -lift LH-> (9) -LH closes, LF opens-> (9) -LF closes->
    stand.  Every impact is a single foot (impact dimf 3, so the switching constraint before it has ns = 3), and two of them
    lift another foot at the same instant.  T = t0 + cycle * (4 swing + 2 ds) with t0 = ds; sto: every event's time is optimised."""
    ev = ContactEvents(phase_dimf=[12], phase_mask=[0b1111])
    t0 = ds
    for k in range(cycle):
        t1 = t0 + k * (2 * ds + 4 * swing)
        ev.push_back(False, t1, 9, sto=sto, post_mask=0b0111)                                           # RH lifts
        ev.push_back(True, t1 + swing, 9, impact_dimf=3, sto=sto, post_mask=0b1011, impact_mask=0b1000)  # RH closes, RF opens
        ev.push_back(True, t1 + 2 * swing, 12, impact_dimf=3, sto=sto, post_mask=0b1111, impact_mask=0b0100)  # RF closes
        ev.push_back(False, t1 + ds + 2 * swing, 9, sto=sto, post_mask=0b1101)                          # LH lifts
        ev.push_back(True, t1 + ds + 3 * swing, 9, impact_dimf=3, sto=sto, post_mask=0b1110, impact_mask=0b0010)  # LH closes, LF opens
        ev.push_back(True, t1 + ds + 4 * swing, 12, impact_dimf=3, sto=sto, post_mask=0b1111, impact_mask=0b0001)  # LF closes
    return ev


def anymal_jump_sto_events() -> ContactEvents:
    """Contact schedule of /root/reference/examples/anymal/jump_sto.cpp:42-48,131-140:
    stand(12) -lift@0.4 (sto)-> flying(0) -impact@0.9 (sto)-> stand; T=1.7."""
    ev = ContactEvents(phase_dimf=[12], phase_mask=[0b1111])
    ev.push_back(False, 0.70 - 0.3, 0, sto=True, post_mask=0)
    ev.push_back(True, 0.70 + 0.30 - 0.1, 12, impact_dimf=12, sto=True, post_mask=0b1111, impact_mask=0b1111)
    return ev
