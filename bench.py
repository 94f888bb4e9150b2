#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json): OCP-iterations/s, ANYmal trot N=40, batch 1024/GPU.

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU algorithm (oracle port, all host threads)
  python bench.py ... --dump-outputs DIR                    also write what the last timed step computed to DIR/*.npy

A "step" is ONE hot-path SQP iteration (SURVEY.md 8d) for every OCP of the batch, given the stage linearisations
resident in HBM:  condense (PDIPM + contact/impact dynamics + SE(3) state-equation correction)  ->  backward Riccati
->  forward Riccati  ->  primal expansion + fraction-to-boundary step sizes  ->  dual expansion + primal/dual update
(the linear-algebra body of OCPSolver::updateSolution, /root/reference/src/solver/ocp_solver.cpp:118-144).
Weak scaling: every GPU owns `--batch` OCPs (instances are independent); with N > 1 the Newton step is all-gathered once
per step over NCCL.  Prints ONE JSON line (rank 0).  PyTorch is plumbing only (streams, events, pinned memory,
torch.distributed).
"""
import argparse
import ctypes
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

N_HORIZON = 40
# Algorithmic bytes per standard stage (doubles -> bytes): SURVEY.md 8(d)'s accounting, applied to what the kernels move today.
BYTES_PER_STAGE_BWD = (3468 + 1776) * 8      # backward reads the 3468-double KKT record, writes P | s | K | k (1776)
BYTES_PER_STAGE_FWD = (3324 + 84) * 8        # forward reads 3324 + writes 84
# condense: 8(d) counts ~2.1k doubles read and ~3.6k written (expansion record) + the 3468-double KKT record (not fused with the
# sweep).  Round 2 no longer stores the acceleration rows of Qafqv / Qafu (1620 -> 648 + 18 doubles): 3.6k -> 2646.
BYTES_PER_STAGE_CONDENSE = (2100 + 2646 + 3468) * 8
BYTES_PER_STAGE_CONDENSE_8D = 46 * 1024      # 8(d)'s literal per-stage figure (without the KKT record), for frac_8d_literal
BYTES_PER_STAGE_MJTJINV = (324 + 216 + 900) * 8               # K1 reads M, J and writes Z
# whole iteration, per standard stage: VERDICT r1's accounting (69.2 + 45.6 + 5 kB = stage layer + sweeps + small records),
# minus the acceleration rows of Qafqv / Qafu that are no longer written by the condensing nor read by the update
BYTES_PER_STAGE_ITERATION = int((69.2 + 45.6 + 5.0) * 1000) - 2 * (1620 - 666) * 8


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes per launch at batch 1024) of the committed `ncu --set full` capture of
    this very command: profiles/r2_final_<kernel>_ncu_summary.txt."""
    path = os.path.join(ROOT, "profiles", f"r2_final_{kernel}_kernel_ncu_summary.txt")
    tot, unit = 0.0, {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
    try:
        for line in open(path):
            f = line.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                tot += float(f[1]) * unit[f[2]]
    except OSError:
        return None, None
    return (tot or None), os.path.relpath(path, ROOT)


FLOP_PER_STAGE_BWD = 285.7e3
FLOP_PER_STAGE_CONDENSE = 300e3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="OCP instances per GPU (BASELINE config 3: 1024)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                    "(float64, at most 64 MB; the inputs are the same on every run)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path: it needs --impl b200")
    return args


DUMP_BYTES = 60 * 10**6  # below 64 MB in all, .npy headers included
DUMP_SEED = 0


def dump_outputs(out_dir, sol, con, direction, steps):
    """The records the timed iteration hands back -- updated solution, updated PDIPM records (slack | dual | residual), Newton
    direction -- of a fixed, seeded sample of the batch's OCPs (as many as fit in DUMP_BYTES), and the primal / dual step sizes
    of every OCP.  ocp_index lists the sampled OCPs."""
    batch = sol.shape[0]
    per_ocp = (sol[0].size + con[0].size + direction[0].size) * 8
    n = min(batch, (DUMP_BYTES - steps.nbytes - batch * 8) // per_ocp)
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(batch, size=n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("solution", sol[idx]), ("constraint_data", con[idx]), ("direction", direction[idx]), ("step_sizes", steps),
                    ("ocp_index", idx)):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def build_problem(batch, seed):
    """Riccati-only inputs (KKT records) -- used by tools/ and the profiling scripts."""
    from helpers import trot_schedule
    from robotoc_b200 import ANYMAL, Layout
    from synth import make_kkt
    dims = ANYMAL
    L = Layout(dims)
    td, ev, ctrl = trot_schedule(N_HORIZON)
    kkt, dx0 = make_kkt(dims, L, ctrl, batch=batch, seed=seed)
    return dims, L, ctrl, kkt, dx0


def build_iteration_problem(batch, seed, getter=None, kgetter=None):
    from helpers import trot_schedule
    from robotoc_b200 import ANYMAL, Layout, StageDims, StageLayout, anymal_constraint_table
    from synth import make_stage_inputs, robotoc_cost_structure
    table = anymal_constraint_table()
    sd = StageDims(ANYMAL, nf_max=12, n_contacts=table.n_contacts, n_box=table.n_box)
    S = StageLayout(sd, getter=getter)
    K = Layout(ANYMAL, getter=kgetter)
    td, ev, ctrl = trot_schedule(N_HORIZON)
    lin, con, sol, dx0 = make_stage_inputs(sd, S, ctrl, batch, seed)
    # inertia matrix / cost Hessians exactly symmetric and structured as robotoc's cost components produce them (Qqq dense; Qvv,
    # Quu, Qff diagonal; Qqv = Qqf = 0), as the reference's containers hold them when the hot path starts
    lin = robotoc_cost_structure(S, lin)
    return dict(dims=ANYMAL, sd=sd, S=S, K=K, table=table, ctrl=ctrl, lin=lin, con=con, sol=sol, dx0=dx0)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
            time.sleep(0.15)  # let nvidia-smi start sampling before the timed region opens
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ts, r in self.rows:
            if t_begin is not None and ts < t_begin:
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


_HOST_CORES = None


def host_cores():
    """Cached: must be taken BEFORE libgomp starts with OMP_PROC_BIND (it pins the calling thread to one place, after which the
    affinity mask of this process reads 1)."""
    global _HOST_CORES
    if _HOST_CORES is None:
        _HOST_CORES = _host_cores()
    return _HOST_CORES


def _host_cores():
    """CPU cores this process may really use: the scheduler affinity mask AND the cgroup CPU quota (a 128-CPU host leased with
    cpu.max = 16 cores only runs 16 threads at a time -- round 1 timed 64 threads there and got a 4x pessimistic baseline)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as fh:
                txt = fh.read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as fh:
                        quota = q / float(fh.read())
            break
        except (OSError, ValueError, IndexError):
            continue
    usable = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return {"logical_cpus": os.cpu_count(), "affinity": aff, "cgroup_quota_cores": quota, "usable": usable}


def _oracle_runner(pr):
    """Returns (cores_info, run): run(mode, nthreads) executes ONE timed pass of the oracle (CPU restatement of the reference
    algorithm) over the whole batch -- condense, Riccati backward + forward, step sizes, update (orc_iteration_batch) -- and
    returns seconds.  Inputs the algorithm mutates in place are restored (untimed) before every pass; only the C call is
    timed.  mode 0: OpenMP over OCP instances ("best-case CPU"); mode 1: one OCP at a time, 4-thread stage loops, serial
    Riccati recursion ("reference-faithful", what robotoc::OCPSolver does with nthreads = 4)."""
    import ctypes as ct
    cores = host_cores()
    # thread placement must be fixed before libgomp starts: one thread per core, neighbours close
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_DYNAMIC", "false")
    import oracle_lib
    lib = oracle_lib.load()
    tmp = tempfile.mkdtemp(prefix="rbt_bench_")
    native = os.path.join(tmp, "liboracle_native.so")
    try:  # -march=native build of the same sources, made on this machine, in a temporary directory
        # -B: always rebuilt -- the build must be tuned for this machine's CPU
        subprocess.run(["make", "-s", "-B", "-C", oracle_lib.ORACLE_DIR, "native", f"NATIVE={native}"], check=True,
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        lib = ct.CDLL(native)
    except Exception:
        pass
    finally:
        shutil.rmtree(tmp, ignore_errors=True)  # a loaded library stays mapped
    from robotoc_b200._lib import rbt_stage_ctrl
    from robotoc_b200.stage import rbt_constraint_table, rbt_stage_dims
    c_int, c_dbl, c_vp = ct.c_int, ct.c_double, ct.c_void_p
    lib.orc_iteration_batch.argtypes = [ct.POINTER(rbt_stage_dims), ct.POINTER(rbt_constraint_table), ct.POINTER(rbt_stage_ctrl),
                                        c_int, c_int, c_dbl] + [c_vp] * 10 + [c_int, c_int]
    S, K, sd, table, ctrl = pr["S"], pr["K"], pr["sd"], pr["table"], pr["ctrl"]
    lin, con0, sol0, dx0 = pr["lin"], pr["con"], pr["sol"], pr["dx0"]
    b, n_grid = lin.shape[0], lin.shape[1]
    kkt = np.zeros((b, n_grid, K.k_stride))
    ex = np.zeros((b, n_grid, S.e_stride))
    ric = np.zeros((b, n_grid, K.r_stride))
    d = np.zeros((b, n_grid, K.d_stride))
    xd = np.zeros((b, n_grid, S.x_stride))
    con, sol = np.empty_like(con0), np.empty_like(sol0)
    steps = np.zeros((b, 2))
    csd = sd.c()
    P = oracle_lib.ptr

    def run(mode, nthreads, nb=None):
        nb = b if nb is None else nb
        np.copyto(con, con0)
        np.copyto(sol, sol0)
        t0 = time.perf_counter()
        info = lib.orc_iteration_batch(ct.byref(csd), ct.byref(table), ctrl, n_grid, nb, 0.1, P(lin), P(con), P(kkt), P(ex), P(ric),
                                       P(dx0), P(d), P(xd), P(sol), P(steps), mode, nthreads)
        el = time.perf_counter() - t0
        assert info == 0
        return el

    return cores, run


WORKLOAD = "anymal_trot_N40 batch={b}/GPU: full hot-path iteration = condense + riccati backward + riccati forward + step sizes + update"
METRIC = "SQP-iterations/s (ANYmal N=40, batch=1024) at 1/2/4/8 B200 vs CPU ref"


def bench_config(batch, n_grid, world, l2_note):
    """The `config` object both arms print (the driver compares them)."""
    return {"workload": WORKLOAD.format(b=batch) + (" + NCCL all-gather of the step (overlapped with the next iteration's condensing / backward sweep)" if world > 1 else ""),
            "n_grid": n_grid, "dims": "nv18 nu12 nx36, 92 inequality rows/stage", "parallelism": f"batch-sharded x{world}",
            "l2": l2_note}


def l2_note(pr):
    lin, K = pr["lin"], pr["K"]
    ws = lin.nbytes + lin.shape[0] * lin.shape[1] * (K.k_stride + K.r_stride) * 8
    return f"per-step working set {ws / 1e9:.2f} GB >> 126 MB L2 (inputs larger than L2; no flush needed)"


def cpu_modes(pr, min_seconds):
    """Both BASELINE.md section 3 modes on the host cores this process may use."""
    cores, run = _oracle_runner(pr)
    b = pr["lin"].shape[0]
    nt = cores["usable"]
    run(0, nt)  # warm-up (page faults of the scratch arrays, libgomp start-up)
    n, el = 0, 0.0
    while el < min_seconds:
        el += run(0, nt)
        n += 1
    best_case = b * n / el
    nb_ref = min(b, 64)  # the serial-in-OCP mode is ~nt/2 times slower: a bounded sample of the same batch
    run(1, 4, nb_ref)
    n1, el1 = 0, 0.0
    while el1 < min_seconds / 3:
        el1 += run(1, 4, nb_ref)
        n1 += 1
    faithful = nb_ref * n1 / el1
    return {"value": best_case, "unit": "OCP-iterations/s", "cores": nt, "kind": "port",
            "sample": f"{n} passes over {b} OCPs, whole iteration per OCP inside one OpenMP loop over OCP instances "
                      f"({nt} threads pinned one per core), {el:.1f} s of CPU-timed work",
            "modes": {"batch_parallel": {"value": best_case, "threads": nt},
                      "reference_faithful": {"value": faithful, "threads": 4, "sample": f"{n1} passes over {nb_ref} OCPs, one OCP at a time, "
                                             "4-thread stage loops, serial Riccati recursion (robotoc::OCPSolver with nthreads = 4)"}},
            "host": cores}


def cpu_leg(pr, min_seconds):
    return cpu_modes(pr, min_seconds)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    host_cores()
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    import oracle_lib
    lib = oracle_lib.load()
    pr = build_iteration_problem(args.batch, 20260927, getter=lib.orc_stage_layout_get, kgetter=lib.orc_layout_get)
    cores, run = _oracle_runner(pr)
    nt = cores["usable"]
    for _ in range(max(args.warmup, 1)):
        run(0, nt)
    el = 0.0
    for _ in range(args.steps):
        el += run(0, nt)
    val = args.batch * args.steps / el
    line = {
        "impl": "reference", "metric": METRIC,
        "value": val, "unit": "OCP-iterations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.batch, len(pr["ctrl"]), max(args.gpus, 1), l2_note(pr)),
        "note": "CPU restatement of the reference algorithm (oracle port pinned against the reference's own Riccati sources, "
                "see tests/test_golden_ref.py; the reference's CMake build needs Eigen3 + Pinocchio, absent here); best-case CPU "
                "mode: OpenMP over OCP instances on every core this process may use",
        "cpu_baseline": {"value": val, "unit": "OCP-iterations/s", "cores": nt, "kind": "port",
                         "sample": f"{args.steps} passes over {args.batch} OCPs", "host": cores},
        "e2e": {"value": val, "unit": "OCP-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    host_cores()
    # (before anything loads libgomp) one OpenMP thread per core, neighbours close: the CPU legs and the parity gate
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    import torch
    import torch.distributed as dist
    from robotoc_b200 import DirectMultipleShooting, RiccatiRecursion
    from robotoc_b200.riccati import DIR
    from robotoc_b200.shard import allgather_step

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: robotoc_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        # one process per GPU on a multi-socket host: run on the CPUs next to this GPU so that the pinned staging buffers of the
        # end-to-end arm are first-touched on the local NUMA node (NVML knows the GPU's CPU affinity)
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        except Exception as e:  # noqa: BLE001  (affinity is an optimisation, never a requirement)
            print(f"[bench] rank {rank}: CPU affinity not set ({e})", file=sys.stderr)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pr = build_iteration_problem(args.batch, 20260927 + rank)
    dims, S, K, ctrl = pr["dims"], pr["S"], pr["K"], pr["ctrl"]
    lin, con, sol, dx0 = pr["lin"], pr["con"], pr["sol"], pr["dx0"]
    n_grid = len(ctrl)
    rr = RiccatiRecursion(dims, n_grid, args.batch, device=local)
    rr.setTimeDiscretization(ctrl)
    dms = DirectMultipleShooting(rr, pr["sd"], pr["table"])
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    lib = rr._lib

    # the Newton step lives in a torch tensor so NCCL can gather it in place
    d_local = torch.zeros((args.batch, n_grid, K.d_stride), dtype=torch.float64, device="cuda")
    rr.bind_buffer(DIR, ctypes.c_void_p(d_local.data_ptr()))
    step_dbl = int(lib.rbt_step_doubles(rr._h))  # dx | du | dlmd,dgmm | dxi | dts,dts_next: the used prefix of a direction record
    d_pack = torch.zeros((args.batch, n_grid, step_dbl), dtype=torch.float64, device="cuda") if world > 1 else None
    d_all = torch.empty((world * args.batch, n_grid, step_dbl), dtype=torch.float64, device="cuda") if world > 1 else None

    # ---- device-resident arm: upload once; every step re-reads the same linearisation / PDIPM / solution records
    dms.condense(lin, con, stream=sp)
    rr.backwardRiccatiRecursion(stream=sp)
    rr.forwardRiccatiRecursion(dx0, stream=sp)
    dms.computeStepSizes(stream=sp)
    dms.integrateSolution(sol, stream=sp)
    torch.cuda.synchronize()
    # ---- parity gate (untimed): EVERY OCP of this rank's batch against the CPU oracle, before anything is timed
    from iteration_check import compare_final, oracle_iteration
    t_chk = time.perf_counter()
    ref = oracle_iteration(pr["sd"], S, K, pr["table"], ctrl, lin, con, sol, dx0,
                           nthreads=max(1, host_cores()["usable"] // max(1, min(world, 8))))
    steps_chk = np.stack([dms.maxPrimalStepSize(sp), dms.maxDualStepSize(sp)], axis=1)
    parity_worst = compare_final(S, K, ctrl, ref, rr.getRiccatiFactorization(sp), d_local.cpu().numpy(), steps_chk,
                                 dms.getSolution(sp), dms.getConstraintData(sp), tol=1e-8)
    print(f"[bench] rank {rank}: parity vs oracle on all {args.batch} OCPs: worst rel err {parity_worst:.2e} "
          f"({time.perf_counter() - t_chk:.1f} s, untimed)", file=sys.stderr, flush=True)
    d_ref_dir = ref["d_upd"]
    del ref
    # the update mutates slack/dual and the solution in place: keep pristine copies and restore them every step (D2D)
    con_dev0, sol_dev0 = torch.from_numpy(con).cuda(), torch.from_numpy(sol).cuda()
    con_work, sol_work = con_dev0.clone(), sol_dev0.clone()
    rr.bind_buffer(7, ctypes.c_void_p(con_work.data_ptr()))
    rr.bind_buffer(9, ctypes.c_void_p(sol_work.data_ptr()))

    NAMES = ["condense_total", "riccati_backward", "riccati_forward", "expand_step_sizes", "update"]

    pending = [False]  # a packed step waits to be gathered

    def gather_pending(ev=None):
        # one NCCL all-gather of the previous iteration's packed step, on its own stream, launched once the condensing of the
        # current iteration has been issued: it then overlaps the (latency / shared-memory bound) backward sweep instead of the
        # HBM-bound condensing kernels
        comm.wait_stream(stream)
        with torch.cuda.stream(comm):
            if ev is not None:
                ev[8].record(comm)
            allgather_step(d_pack, out=d_all)
            if ev is not None:
                ev[6].record(comm)
        pending[0] = False

    def step(ev=None):
        # restore what the iteration mutates in place -- slack | dual of the PDIPM records and the solution records -- so that
        # every timed step computes the same, oracle-checked iteration (D2D, outside the per-kernel event pairs but inside the
        # step time; a real SQP loop has no such copy)
        con_work[:, :, :2 * S.ncp].copy_(con_dev0[:, :, :2 * S.ncp])
        sol_work.copy_(sol_dev0)
        calls = [lambda: dms.condense(stream=sp), lambda: rr.backwardRiccatiRecursion(stream=sp),
                 lambda: rr.forwardRiccatiRecursion(stream=sp), lambda: dms.computeStepSizes(stream=sp),
                 lambda: dms.integrateSolution(stream=sp)]
        for k, call in enumerate(calls):
            if ev is not None:
                ev[k].record(stream)
                if k == 0:  # rbt_condense = MJtJinv kernel + condensing kernel: an event between them splits the two
                    ev[7].record(stream)  # (creates the handle)
                    lib.rbt_set_condense_event(rr._h, ctypes.c_void_p(ev[7].cuda_event))
            call()
            if ev is not None and k == 0:
                lib.rbt_set_condense_event(rr._h, None)
            if world > 1 and k == 0 and pending[0]:
                gather_pending(ev)
        if ev is not None:
            ev[len(calls)].record(stream)
        if world > 1:
            stream.wait_stream(comm)  # the previous gather has finished reading the pack buffer
            rc = lib.rbt_pack_step(rr._h, ctypes.c_void_p(d_pack.data_ptr()), sp)
            assert rc == 0, rr._err()
            pending[0] = True

    comm = torch.cuda.Stream() if world > 1 else None
    for _ in range(max(args.warmup, 3)):
        step()
    if world > 1:
        gather_pending()
    torch.cuda.synchronize()
    l0 = rr.launch_count()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(9)] for _ in range(args.steps)]
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clk = ClockSampler(local)
    if rank == 0 and not os.environ.get("RBT_BENCH_NO_CLOCKS"):
        clk.start()  # (sleeps ~0.15 s while nvidia-smi spins up: must happen BEFORE the barrier that aligns the ranks)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_host0 = time.perf_counter()
    t_beg.record(stream)
    for k in range(args.steps):
        step(evs[k])
    if world > 1:
        gather_pending()          # the last step's gather is inside the timed region
        stream.wait_stream(comm)
    t_end.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = clk.stop(t_host0) if rank == 0 else None
    launches = rr.launch_count() - l0
    ms = t_beg.elapsed_time(t_end)
    kms = {n: float(np.mean([e[k].elapsed_time(e[k + 1]) for e in evs])) for k, n in enumerate(NAMES)}
    kms["mjtjinv"] = float(np.mean([e[0].elapsed_time(e[7]) for e in evs]))
    kms["condense"] = float(np.mean([e[7].elapsed_time(e[1]) for e in evs]))
    if world > 1:
        kms["nccl_allgather_step"] = float(np.mean([e[8].elapsed_time(e[6]) for e in evs[1:]]))  # on the comm stream (steps 2..K)
    print(f"[bench] rank {rank}: {ms / args.steps:.3f} ms/step on its own device clock", file=sys.stderr, flush=True)
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    assert int(rr.info().max()) == 0, "Cholesky failure flagged on device"
    if world > 1:  # config 5: this rank's shard of the gathered step is the step the oracle computes for these OCPs
        shard = d_all[rank * args.batch:(rank + 1) * args.batch].cpu().numpy()
        nxu = min(K.d_dxi, step_dbl)
        err = np.max(np.abs(shard[..., :nxu] - d_ref_dir[..., :nxu])) / np.max(np.abs(d_ref_dir[..., :nxu]))
        assert err < 1e-8, f"rank {rank}: gathered step disagrees with the oracle ({err:.2e})"
    sol_dev = dms.getSolution()
    steps_dev = np.stack([dms.maxPrimalStepSize(), dms.maxDualStepSize()], axis=1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sol_dev, dms.getConstraintData(), d_local.cpu().numpy(), steps_dev)

    # ---- end-to-end arm: host (pinned) buffers through the one-call C-ABI entry point, H2D + D2H inside the timed region
    pin = lambda a: torch.from_numpy(a).pin_memory()  # noqa: E731
    lin_p, con_p, sol_p, dx0_p = pin(lin), pin(con), pin(sol), pin(dx0)
    sol_o = torch.zeros(sol.shape, dtype=torch.float64).pin_memory()
    con_o = torch.from_numpy(con.copy()).pin_memory()  # slack | dual are refreshed by the call
    steps_o = torch.empty((args.batch, 2), dtype=torch.float64).pin_memory()
    P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731

    # the host adaptor's output format: packed upper triangles of the symmetric blocks (include/rbt_stage_layout.h), made
    # once outside the timed region -- it is what the host side hands over, like the records themselves
    dms.setWireCostStructure(True)
    wire_p = pin(dms.pack_wire(lin))
    e2e_mode = os.environ.get("RBT_E2E_MODE", "resident")  # resident | wire | dense
    use_wire = e2e_mode != "dense"
    res_p = pin(np.ascontiguousarray(con[:, :, S.c_res:S.c_res + S.ncp]))
    sd_o = torch.zeros((args.batch, n_grid, 2 * S.ncp), dtype=torch.float64).pin_memory()

    def e2e_step():
        if e2e_mode == "resident":
            # the solver state (solution, slack, dual) lives on the device, as OCPSolver keeps s_ and the constraint data
            # between iterations; only what the host recomputes at a new linearisation point crosses PCIe.  (The D2D restore
            # of the state is a bench artefact -- every timed step then computes the same, oracle-checked iteration.)
            con_work[:, :, :2 * S.ncp].copy_(con_dev0[:, :, :2 * S.ncp])
            sol_work.copy_(sol_dev0)
            rc = lib.rbt_iteration_host_resident(rr._h, P(wire_p), P(lin_p), P(res_p), P(dx0_p), P(sol_o), P(sd_o), P(steps_o), sp)
        elif use_wire:
            rc = lib.rbt_iteration_host_wire(rr._h, P(wire_p), P(lin_p), P(con_p), P(sol_p), P(dx0_p), P(sol_o), P(con_o),
                                             P(steps_o), sp)
        else:
            rc = lib.rbt_iteration_host(rr._h, P(lin_p), P(con_p), P(sol_p), P(dx0_p), P(sol_o), P(con_o), P(steps_o), sp)
        assert rc == 0, rr._err()

    e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_beg.record(stream)
    for _ in range(args.e2e_steps):
        e2e_step()
    e_end.record(stream)
    torch.cuda.synchronize()
    e2e_ms = e_beg.elapsed_time(e_end)
    if world > 1:
        tt = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt.item())
    # what the call actually moves (padding / unused sections never cross PCIe)
    h2d, d2h = dms.iteration_host_bytes(wire=use_wire, resident=(e2e_mode == "resident"))
    used = dms.layout.s_xi + dms.layout.nsm
    assert np.array_equal(sol_o.numpy()[:, :, :used], sol_dev[:, :, :used]) and np.array_equal(steps_o.numpy(), steps_dev), \
        "e2e path disagrees with the device-resident path"

    if rank == 0:
        peak, peak_src = peaks()
        units = args.batch * N_HORIZON                       # standard stages per launch (SURVEY.md 8d)
        dom = max((k for k in kms if k != "condense_total"), key=kms.get)
        alg_bytes = {"riccati_backward": BYTES_PER_STAGE_BWD, "riccati_forward": BYTES_PER_STAGE_FWD,
                     "condense": BYTES_PER_STAGE_CONDENSE}.get(dom, BYTES_PER_STAGE_BWD) * units
        ach = alg_bytes / (kms[dom] * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic(dom) if dom in ("condense", "riccati_backward") else (None, None)
        kname = {"riccati_backward": "riccati_backward_kernel<18,12,12>", "condense": "condense_kernel<18,12,12>",
                 "riccati_forward": "riccati_forward_kernel<18,12,12>"}.get(dom, dom)
        line = {
            "metric": METRIC,
            "value": world * args.batch * args.steps / (ms * 1e-3), "unit": "OCP-iterations/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(args.batch, n_grid, world, l2_note(pr)),
            "clocks": clocks, "gpu_launches": int(launches),
            "parity": {"checked_ocps": args.batch, "worst_rel_err_vs_oracle": parity_worst, "tol": 1e-8},
            "kernels_ms": kms,
            "riccati_only": {"value": world * args.batch / ((kms["riccati_backward"] + kms["riccati_forward"]) * 1e-3),
                             "unit": "OCP-iterations/s", "note": "backward + forward sweeps only (the parity-checked core, 8d)"},
            "e2e": {"value": world * args.batch * args.e2e_steps / (e2e_ms * 1e-3), "unit": "OCP-iterations/s",
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps,
                    "api": {"resident": "rbt_iteration_host_resident (pinned host buffers: wire linearisation records -- packed symmetric "
                                        "blocks, contact blocks sized by the active contacts, cost Hessians as robotoc's cost components produce "
                                        "them (Qqq dense; Qvv, Quu, Qff diagonal) -- PDIPM residuals, dx0 in; solution, "
                                        "slack|dual, step sizes out; solver state resident on the device; 8-chunk "
                                        "upload/compute/download pipeline)",
                            "wire": "rbt_iteration_host_wire (as resident, plus PDIPM slack|dual and the solution uploaded every step)",
                            "dense": "rbt_iteration_host (dense linearisation records)"}[e2e_mode]},
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": (traffic * args.batch / 1024) if traffic else None,
                         "traffic_source": f"dram__bytes_read + write of the ncu --set full capture of this command ({traffic_src}), per launch",
                         "frac_8d_literal": (BYTES_PER_STAGE_CONDENSE_8D * units / (kms[dom] * 1e-3) / 1e9 / peak) if dom == "condense" else None,
                         "iteration": {"algorithmic_bytes": BYTES_PER_STAGE_ITERATION * units,
                                       "achieved": BYTES_PER_STAGE_ITERATION * units / (ms / args.steps * 1e-3) / 1e9,
                                       "frac": BYTES_PER_STAGE_ITERATION * units / (ms / args.steps * 1e-3) / 1e9 / peak},
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                         "per_kernel_GBps": {
                             "riccati_backward": BYTES_PER_STAGE_BWD * units / (kms["riccati_backward"] * 1e-3) / 1e9,
                             "riccati_forward": BYTES_PER_STAGE_FWD * units / (kms["riccati_forward"] * 1e-3) / 1e9,
                             "condense": BYTES_PER_STAGE_CONDENSE * units / (kms["condense"] * 1e-3) / 1e9,
                             "mjtjinv": BYTES_PER_STAGE_MJTJINV * units / (kms["mjtjinv"] * 1e-3) / 1e9},
                         "fp64_tflops": {"riccati_backward": FLOP_PER_STAGE_BWD * units / (kms["riccati_backward"] * 1e-3) / 1e12,
                                         "condense": FLOP_PER_STAGE_CONDENSE * units / (kms["condense"] * 1e-3) / 1e12},
                         "fp64_peak_tflops": 37.1},
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_leg(pr, min_seconds=10.0)
        print(json.dumps(line), flush=True)
    rr.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
