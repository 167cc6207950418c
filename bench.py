#!/usr/bin/env python
"""bench.py -- batched OCP SQP solves/sec (H=20 quadrotor MPC) on N B200s, one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one batched CUDA_SQP solve of B instances per GPU (BASELINE.json configs[2]:
quadrotor nx=12 nu=4 H=20, B=4096 random initial states, SQP_step alpha=0.1, ADMM_step
step_num=10, OSQP settings of SQPOptimizationSolver.cpp:81-85), every step from the same cold
iterate x=0 so that all steps do identical work.

  value   solves/s, whole job, inputs resident in HBM, CUDA events around ocp_b200_solve_batch_device
  e2e     same through ocp_b200_solve_batch with pinned HOST buffers (H2D + D2H inside the timed region)
  roofline  the ADMM kernel: `frac` = SURVEY.md §8d's streaming byte count (with the iteration / solve / check counts
            of the stats buffer) over its CUDA-event time and the measured HBM peak -- an EFFECTIVE rate: the kernel keeps
            its state on chip and in L2 and is bound by dependent-instruction latency (frac_dram, counters alongside)
  secondary  with 2 or more GPUs (or --secondary): BASELINE.json configs[3] / [4] at their stated TOTAL sizes, split over
            the ranks (strong scaling), one timed step each
  cpu_baseline  the oracle (restated reference CPU path) on the host cores, bounded sample

`--impl reference` times the oracle alone (rank 0 only).  torch is used for device memory,
streams, events and torch.distributed -- not for compute.

`--dump-outputs DIR` writes what the last timed step returned (x [B, N], f [B], stats [B, 12], gathered over the
ranks) as DIR/<name>.npy in float64, so that two builds can be compared output for output on the same seeded inputs.

The bench writes nothing into the source tree (it may be read-only): stage libraries are looked up in, and if
missing compiled into, a temporary directory (see private_share_dir).
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

# stdout carries exactly one JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints
# its version banner there), so fd 1 is pointed at stderr for the duration of the run and the line is written
# to the saved descriptor.
_RESULT_FD = None


def capture_stdout():
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.dont_write_bytecode = True     # no __pycache__ in the tree for the modules imported from it

METRIC = "batched OCP SQP solves/sec (H=20)"
UNIT = "solves/s"
SEED = 0xB200 + 2          # SURVEY.md §8d: 0xB200 + config index
PROBLEM = "quadrotor"
ALPHA, STEP_NUM = 0.1, 10


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU (weak scaling); default 4096 (quadrotor), 592 otherwise")
    ap.add_argument("--workload", default="quadrotor", choices=sorted(WORKLOADS),
                    help="quadrotor = the configuration the metric is quoted on (default); the others are BASELINE.json's "
                         "larger shapes, not bench lines of record")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="solves in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--latency-solves", type=int, default=50)
    ap.add_argument("--secondary", default="auto", choices=["auto", "on", "off"],
                    help="bounded pass over BASELINE.json configs[3]/[4] at their stated total sizes (auto: with >= 2 GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write x, f and stats of the last timed step as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


WORKLOADS = {
    "quadrotor": ("quadrotor MPC nx=12 nu=4 H=20 dt=0.005, multiple shooting RK4", "BASELINE.json configs[2]", 20),
    "cartpole": ("cart-pole swing-up nx=4 nu=1 H=200 dt=0.01, multiple shooting RK4", "BASELINE.json configs[4]", 200),
    "centroidal": ("centroidal legged-robot MPC nx=24 nu=12 H=50 dt=0.01 with friction pyramids", "BASELINE.json configs[3]", 50),
}


def select_workload(args):
    """The default is the configuration the metric is quoted on; --workload switches the module constants."""
    global PROBLEM, METRIC
    PROBLEM = args.workload
    METRIC = f"batched OCP SQP solves/sec (H={WORKLOADS[PROBLEM][2]})"
    if args.batch <= 0:
        args.batch = 4096 if PROBLEM == "quadrotor" else 592


def initial_iterate(frames, horizon):
    """Cold iterate x = 0 for the quadrotor (as the reference starts); the other shapes start from the initial
    frame held over the horizon (x = 0 makes the first cart-pole QP primal infeasible)."""
    x0 = np.tile(frames, (1, horizon))
    if PROBLEM == "quadrotor":
        x0[:] = 0.0
    return x0


def workload_config(batch, n_gpus):
    desc, cfg, _ = WORKLOADS[PROBLEM]
    return {"workload": f"{desc}, {batch} random initial states per GPU ({cfg})",
            "solve_method": "CUDA_SQP", "SQP_step": ALPHA, "ADMM_step": STEP_NUM, "eps_abs": 1e-3, "eps_rel": 1e-3,
            "admm_max_iter": 10000, "batch_per_gpu": batch, "parallelism": f"instances sharded over {n_gpus} GPU(s), no data-path collective",
            "l2": "flushed between timed steps (256 MiB write); per-step QP buffers (163 MB at B=4096) also exceed L2"}


# ---------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_run(sample: int, threads: int, repeats: int = 1, warmup: int = 0, reuse_symbolic: bool = False):
    import _oracle
    ora = _oracle.OracleProblem(PROBLEM, alpha=ALPHA, step_num=STEP_NUM)
    if reuse_symbolic:   # variant without the reference's per-step symbolic re-setup (SURVEY.md 8d)
        ora.set_schedule(STEP_NUM, ALPHA, reuse_symbolic=True)
    frames, refs = ora.sample_inputs(sample, SEED)
    x0 = initial_iterate(frames, ora.horizon)
    times = []
    for it in range(warmup + repeats):
        t0 = time.perf_counter()
        ora.solve_batch(frames, refs, x0=x0, nthreads=threads)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return times


def cpu_latency_p50(solves: int):
    """p50 wall time of single-instance solves on one host thread (SURVEY.md 8d: latency of the CPU path)."""
    import _oracle
    ora = _oracle.OracleProblem(PROBLEM, alpha=ALPHA, step_num=STEP_NUM)
    frames, refs = ora.sample_inputs(solves, SEED)
    x0 = initial_iterate(frames, ora.horizon)
    ms = []
    for i in range(solves):
        t0 = time.perf_counter()
        ora.solve_batch(frames[i:i + 1], refs[i:i + 1], x0=x0[i:i + 1], nthreads=1)
        ms.append(1e3 * (time.perf_counter() - t0))
    return {"p50_ms": float(np.median(ms)), "solves": solves}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    sample = args.cpu_sample or (max(64, 32 * threads) if PROBLEM == "quadrotor" else 2 * threads)
    times = cpu_run(sample, threads, repeats=args.steps, warmup=args.warmup)
    total = sum(times)
    value = sample * args.steps / total
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "reference", "config": workload_config(args.batch, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{sample} of the workload's instances per step, one instance per host thread at a time; "
                                       "oracle = FP64 restatement of the reference's CPU SQP+OSQP path (CasADi/OSQP are not "
                                       "installable here), cold OSQP set-up every SQP step like the reference"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1] or [r for (_, r) in self.rows]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# files: stage libraries and dumped outputs
# ---------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64_000_000


def private_share_dir():
    """Problem() needs a writable share directory for its generated stage library.  Unless OCP_B200_SHARE_DIR names
    one, the bench uses a temporary directory (removed at exit) in which the stage libraries build() left in the
    package are linked, so that a model built there is not compiled again and the tree is never written to."""
    if os.environ.get("OCP_B200_SHARE_DIR"):
        return
    share = Path(tempfile.mkdtemp(prefix="ocp_b200_bench_"))
    atexit.register(shutil.rmtree, share, True)
    (share / "code_gen").mkdir()
    for so in (ROOT / "optimal_control_problem_b200" / "share" / "code_gen").glob("*.so"):
        (share / "code_gen" / so.name).symlink_to(so)
    os.environ["OCP_B200_SHARE_DIR"] = str(share)


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes every array as out_dir/<name>.npy in float64.  The arrays share their leading (instance) axis; when the
    files would exceed DUMP_LIMIT_BYTES together, each keeps the same fixed, seeded sample of instances."""
    rows = next(iter(arrays.values())).shape[0]
    total = sum(8 * a.size for a in arrays.values())
    room = DUMP_LIMIT_BYTES - 1024 * len(arrays)       # .npy headers are 128 bytes each
    if total > room:
        keep = room * rows // total
        idx = np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        print(f"bench.py: outputs exceed {DUMP_LIMIT_BYTES / 1e6:.0f} MB, kept {keep} of {rows} instances (seed 0)",
              file=sys.stderr)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out / f"{k}.npy", np.ascontiguousarray(a, dtype=np.float64))


# ---------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------
def algorithmic_bytes(dims, nnz_pu, stats, ocp, direct=None):
    """SURVEY.md 8(d), as written: bytes one batched solve (all its SQP steps) moves if every operand of every operation
    is streamed once (no credit for shared-memory residency), with the ACTUAL counts of the stats buffer:
        bytes_admm(K) = 8 [ (K+1)(nnzPu + 2 nnzA) + 2 nnzA + (6K+8) n + (2K+12) m ]      per ADMM iteration, K = KKT solves / iteration
        bytes_check   = 8 [ nnzPu + 2 nnzA + 4n + 4m ]                                    per residual check
    (K = 1 for the direct LDL' kernel: one application of the factor per iteration.)  Returns (contract bytes, counts,
    direct-model bytes or None).  The direct model (DESIGN.md 5.3, round 1's figure) counts what the block LDL' reads --
    dense factor blocks instead of PCG operator applications, plus the set-up -- and is kept for comparison only."""
    n, m, nnz_a = dims["n"], dims["m"], dims["nnz_a"]
    iters = stats[:, ocp.STAT["admm_iters"]].sum()
    solves = stats[:, ocp.STAT["pcg_iters"]].sum()
    checks = stats[:, ocp.STAT["checks"]].sum()
    qps = stats[:, ocp.STAT["sqp_steps"]].sum()
    mat = nnz_pu + 2 * nnz_a
    contract = 8.0 * ((solves + iters) * mat + iters * (2 * nnz_a + 8 * n + 12 * m) + solves * (6 * n + 2 * m)) \
        + 8.0 * checks * (mat + 4 * n + 4 * m)
    counts = dict(admm_iters=float(iters), kkt_solves=float(solves), checks=float(checks), qps=float(qps),
                  K=float(solves / max(iters, 1.0)))
    model = None
    if direct is not None:
        np_, bs, nb = direct["np"], direct["bs"], direct["nb"]
        fac = nb * bs * bs + 2 * (nb - 1) * bs * bs + 2 * np_ * nb * bs + np_ * np_
        per_iter = 8.0 * (2 * nnz_a + fac + 10 * n + 9 * m)
        setup = 8.0 * ((nnz_a + nnz_pu + n + 2 * m) + 10 * 3 * (2 * nnz_pu + nnz_a) + 4 * fac)
        model = iters * per_iter + qps * setup + 8.0 * checks * (mat + 4 * n + 4 * m)
    return contract, counts, model


def secondary_pass(ocp, torch, dist, world, rank, local, dev):
    """BASELINE.json configs[3] (16 384 centroidal instances) and configs[4] (65 536 cart-pole instances) at their stated
    TOTAL sizes, split evenly over the ranks (strong scaling), one warm-up and one timed batched solve each, device-timed
    with the gather of solutions and statistics inside; max over ranks."""
    from optimal_control_problem_b200.sharding import gather_shards
    out = []
    for name, total, cfg in (("centroidal", 16384, "BASELINE.json configs[3]"), ("cartpole", 65536, "BASELINE.json configs[4]")):
        Bk = total // world
        prob = ocp.Problem(name, alpha=ALPHA, step_num=STEP_NUM)
        sol = ocp.Solver.create(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, prob.a_colptr, prob.a_rowidx,
                                settings=prob.get_settings(), np_=prob.np_, nf=prob.nf, horizon=prob.horizon,
                                model_library=prob.model_library, device=local)
        frames_h, refs_h = prob.sample_inputs(Bk, SEED + 7 + 1000 * rank)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        d_frames, d_p, d_lbx, d_ubx, d_lbg, d_ubg = t(frames_h), t(refs_h), t(prob.lbx), t(prob.ubx), t(prob.lbg), t(prob.ubg)
        d_x0 = t(np.tile(frames_h, (1, prob.horizon)))
        d_x = torch.zeros(Bk, prob.N, dtype=torch.float64, device=dev)
        d_f = torch.zeros(Bk, dtype=torch.float64, device=dev)
        d_st = torch.zeros(Bk, ocp.NSTATS, dtype=torch.float64, device=dev)
        stream = torch.cuda.current_stream()
        ms = 0.0
        for it in range(2):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            d_x.copy_(d_x0)
            sol.solve_batch_device(Bk, d_frames.data_ptr(), d_p.data_ptr(), d_lbx.data_ptr(), d_ubx.data_ptr(), d_lbg.data_ptr(),
                                   d_ubg.data_ptr(), d_x.data_ptr(), d_f.data_ptr(), d_st.data_ptr(), stream.cuda_stream)
            if world > 1:
                gather_shards(d_x, world * Bk); gather_shards(d_st, world * Bk)
            e1.record(stream)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
        tm = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        st = d_st.cpu().numpy()
        out.append({"workload": f"{WORKLOADS[name][0]} ({cfg})", "total_instances": world * Bk, "instances_per_gpu": Bk,
                    "scaling": "strong", "value": world * Bk / (float(tm.item()) * 1e-3), "unit": UNIT,
                    "ms_per_step": float(tm.item()), "steps": 1, "warmup": 1,
                    "admm_iters_per_solve": float(st[:, ocp.STAT["admm_iters"]].mean()),
                    "solved_fraction_rank0": float((st[:, ocp.STAT["qp_status"]] == ocp.QP_SOLVED).mean()),
                    "plan": sol.launch_plan()["wide"]})
        sol.close()
        del d_x, d_x0, d_st, d_f
        torch.cuda.empty_cache()
    return out


def b200_arm(args):
    import torch
    import torch.distributed as dist

    private_share_dir()                  # before the package reads OCP_B200_SHARE_DIR
    import optimal_control_problem_b200 as ocp
    from optimal_control_problem_b200.sharding import gather_shards

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device visible and there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    B = args.batch

    prob = ocp.Problem(PROBLEM, alpha=ALPHA, step_num=STEP_NUM)
    # one handle per (process, device): the problem's own handle lives on device 0 of the process's
    # view, so create the handle explicitly on this rank's device
    sol = ocp.Solver.create(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, prob.a_colptr, prob.a_rowidx,
                            settings=prob.get_settings(), np_=prob.np_, nf=prob.nf, horizon=prob.horizon,
                            model_library=prob.model_library, device=local)
    dims = prob.dims
    nnz_pu = int(sum(1 for j in range(prob.n) for k in range(prob.h_colptr[j], prob.h_colptr[j + 1]) if prob.h_rowidx[k] <= j))

    frames_h, refs_h = prob.sample_inputs(B, SEED + 1000 * rank)
    f64 = dict(dtype=torch.float64, device=dev)
    d_frames = torch.from_numpy(frames_h).to(dev); d_p = torch.from_numpy(refs_h).to(dev)
    d_lbx = torch.from_numpy(prob.lbx).to(dev); d_ubx = torch.from_numpy(prob.ubx).to(dev)
    d_lbg = torch.from_numpy(prob.lbg).to(dev); d_ubg = torch.from_numpy(prob.ubg).to(dev)
    x0_h = initial_iterate(frames_h, prob.horizon)
    d_x0 = torch.from_numpy(x0_h).to(dev)
    d_x = torch.zeros(B, prob.N, **f64); d_f = torch.zeros(B, **f64); d_stats = torch.zeros(B, ocp.NSTATS, **f64)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    gathered = {}
    stream = torch.cuda.current_stream()

    def device_step():
        d_x.copy_(d_x0)
        sol.solve_batch_device(B, d_frames.data_ptr(), d_p.data_ptr(), d_lbx.data_ptr(), d_ubx.data_ptr(),
                               d_lbg.data_ptr(), d_ubg.data_ptr(), d_x.data_ptr(), d_f.data_ptr(), d_stats.data_ptr(),
                               stream.cuda_stream)
        if world > 1:  # the one collective of the path: gather solutions and statistics (SURVEY.md §8e)
            gathered["x"] = gather_shards(d_x, world * B)
            gathered["stats"] = gather_shards(d_stats, world * B)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident inputs ------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        device_step()
    barrier()
    launches0 = sol.launch_count()
    sol.set_profiling(True)
    sol.get_profile(reset=True)
    sampler = ClockSampler(local) if rank == 0 else None
    t_wall0 = time.perf_counter()
    step_ms = []
    for _ in range(args.steps):
        flush.fill_(1)                                   # L2 flush, outside the event pair
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        device_step()
        e1.record(stream)
        barrier()
        step_ms.append(e0.elapsed_time(e1))
    t_wall1 = time.perf_counter()
    if args.dump_outputs:                                # what the last timed step returned, before anything else runs
        outputs = {"x": gathered.get("x", d_x), "f": gather_shards(d_f, world * B), "stats": gathered.get("stats", d_stats)}
        outputs = {k: v.cpu().numpy() for k, v in outputs.items()}
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    prof = sol.get_profile(reset=True)
    sol.set_profiling(False)
    launches = sol.launch_count() - launches0
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    value = world * B * args.steps / (total_ms * 1e-3)

    stats_h = d_stats.cpu().numpy()
    solved = int((stats_h[:, ocp.STAT["qp_status"]] == ocp.QP_SOLVED).sum())
    dd = sol.device_dims()
    plan = sol.launch_plan()
    direct = dict(np=plan["tri_np"], bs=plan["tri_bs"], nb=plan["tri_nb"]) if plan["tri_ok"] else None   # from the handle
    bytes_per_solve_call, counts, model_bytes = algorithmic_bytes(dims, nnz_pu, stats_h, ocp, direct)
    admm_ms_per_launch = prof["admm"]["ms"] / max(1, prof["admm"]["launches"])
    bytes_per_launch = bytes_per_solve_call / STEP_NUM
    achieved = bytes_per_launch / (admm_ms_per_launch * 1e-3) / 1e9 if admm_ms_per_launch > 0 else 0.0
    model_achieved = (model_bytes / STEP_NUM) / (admm_ms_per_launch * 1e-3) / 1e9 if model_bytes and admm_ms_per_launch > 0 else None
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak, peak_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    # DRAM traffic and issue / occupancy counters of the same kernel from the committed ncu capture (profiles/)
    traffic, counters = None, None
    tpath = ROOT / "profiles" / "admm_traffic.json"
    if tpath.exists() and PROBLEM == "quadrotor":
        tj = json.loads(tpath.read_text())
        traffic = tj.get("dram_bytes_per_launch")
        counters = tj.get("counters")

    # ---- e2e: pinned host buffers through ocp_b200_solve_batch -----------------------------------
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    hp_frames, hp_refs = pin(frames_h), pin(refs_h)
    hp_x = torch.zeros(B, prob.N, dtype=torch.float64).pin_memory()
    hp_f = torch.zeros(B, dtype=torch.float64).pin_memory()
    hp_st = torch.zeros(B, ocp.NSTATS, dtype=torch.float64).pin_memory()
    nx, nf_, nst = hp_x.numpy(), hp_f.numpy(), hp_st.numpy()

    def host_step():
        nx[:] = x0_h
        sol.solve_batch(hp_frames.numpy(), hp_refs.numpy(), prob.lbx, prob.ubx, prob.lbg, prob.ubg, nx, nf_, nst)

    for _ in range(2):
        host_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        host_step()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(e2e_s.item())
    h2d = 8 * (B * (prob.nf + prob.np_ + prob.N) + 2 * prob.N + 2 * prob.ng)
    d2h = 8 * B * (prob.N + 1 + ocp.NSTATS)
    e2e_match = float(np.abs(nx - d_x.cpu().numpy()).max())

    # ---- p50 single-solve latency (B = 1, host API) ----------------------------------------------
    lat = []
    if rank == 0 and args.latency_solves > 0:
        x1 = np.zeros((1, prob.N)); f1 = np.zeros(1)
        for i in range(args.latency_solves + 5):
            x1[:] = x0_h[i % B]
            t0 = time.perf_counter()
            sol.solve_batch(frames_h[i % B:i % B + 1], refs_h[i % B:i % B + 1], prob.lbx, prob.ubx, prob.lbg, prob.ubg, x1, f1)
            if i >= 5:
                lat.append(1e3 * (time.perf_counter() - t0))

    # ---- CPU baseline on rank 0 at N = 1 ----------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        sample = args.cpu_sample or (max(64, 128 * threads) if PROBLEM == "quadrotor" else 2 * threads)   # ~25 core-seconds
        t = cpu_run(sample, threads, repeats=1, warmup=0)[0]
        t1 = cpu_run(min(sample, 32), 1, repeats=1, warmup=0)[0] / min(sample, 32)
        p50_1t = cpu_latency_p50(200 if PROBLEM == "quadrotor" else 8)
        tr = cpu_run(sample, threads, repeats=1, warmup=0, reuse_symbolic=True)[0]
        cpu = {"value": sample / t, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{sample} instances of the same workload (first of the {B}), one instance per host thread at a time, "
                         f"{t:.1f} s wall; single-thread {1e3 * t1:.1f} ms/solve; restated reference CPU path (cold OSQP "
                         f"set-up every SQP step), value_without_resetup keeps ordering + elimination tree between steps",
               "single_thread_ms_per_solve": 1e3 * t1, "single_thread_p50_ms": p50_1t["p50_ms"],
               "single_thread_p50_solves": p50_1t["solves"], "value_without_resetup": sample / tr}

    # ---- BASELINE.json configs[3] / [4] at their stated total sizes (strong scaling over the ranks) ------------
    secondary = None
    if PROBLEM == "quadrotor" and (args.secondary == "on" or (args.secondary == "auto" and world >= 2)):
        del flush
        torch.cuda.empty_cache()
        secondary = secondary_pass(ocp, torch, dist, world, rank, local, dev)

    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "impl": "b200", "config": workload_config(B, world),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "max_abs_diff_vs_device_path": e2e_match},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic,
                             "kernel": {4: "admm_compact_kernel", -1: "admm_solve_kernel (PCG)"}.get(plan["wide"]["place"], "admm_direct_kernel"),
                             "peak_source": peak_src,
                             "formula": "SURVEY.md 8(d): iters*bytes_admm(K) + checks*bytes_check, K = kkt_solves/admm_iters from the stats buffer",
                             "limiter": "dependent-instruction latency: per-instance state lives in shared memory and an L2-resident slab, "
                                        "`achieved` is an effective (algorithmic) rate, not DRAM utilisation",
                             "achieved_dram": (traffic / (admm_ms_per_launch * 1e-3) / 1e9) if traffic and admm_ms_per_launch > 0 else None,
                             "frac_dram": (traffic / (admm_ms_per_launch * 1e-3) / 1e9 / peak) if traffic and admm_ms_per_launch > 0 else None,
                             "frac_direct_model": (model_achieved / peak) if model_achieved else None,
                             "counters": counters,
                             "algorithmic_bytes_per_launch": bytes_per_launch, "kernel_ms_per_launch": admm_ms_per_launch,
                             "kernel_share_of_step": prof["admm"]["ms"] / max(total_ms, 1e-9),
                             "assemble_ms_per_launch": prof["assemble"]["ms"] / max(1, prof["assemble"]["launches"]),
                             "counts_per_batched_solve": counts},
                "cpu_baseline": cpu,
                "clocks": clocks,
                "latency_p50_ms": float(np.median(lat)) if lat else None,
                "solved_fraction": solved / B,
                "device": torch.cuda.get_device_name(local),
                "kernel_plan": dict(dd, linsys="block-tridiagonal LDL' (direct)" if direct else "PCG", wide=plan["wide"], deep=plan["deep"],
                                    tri=direct)}
        if secondary is not None:
            line["secondary"] = secondary
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    select_workload(args)
    capture_stdout()
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
