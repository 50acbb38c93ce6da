#!/usr/bin/env python3
"""bench.py -- PDHG iterations/s of the B200 PDLP engine on BASELINE.json's synthetic LPs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload S3|S2|S5] [--impl ours|reference] [--dump-outputs DIR]

A "step" is ONE PDHG iteration of the hot path (primal step, A x + dual step, A'y +
step rule) on the stated LP; the timed region runs exactly K iterations INCLUDING the
check iterations (average iterate, 2 extra SpMV, residuals, restarts) that fall inside
them, with the LP resident in HBM (`value`), and the same K iterations through the
public host-buffer call b200pdlp_solve -- formulate + scale + layout + H2D + K
iterations + D2H of the HighsSolution -- (`e2e`).  N > 1: the same LP row-partitioned
over N GPUs, one process per GPU (torchrun), reduce-scatter of A'y + all-gather of x per iteration
(fused into the engine's own kernels over NVLink peer memory; B200PDLP_NO_P2P=1 selects NCCL)
("strong" scaling: total work is fixed).  Prints ONE JSON line on rank 0.

--impl reference times the reference's own CPU pdlp (oracle/_ref, the unmodified HiGHS
built by oracle/build_ref.py) on the same LP on the host cores (it is single-threaded),
steady-state iterations/s from a two-point fit so that the O(nnz) setup drops out.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep stdout to the one JSON line (NCCL prints its version banner at INFO/VERSION)

import numpy as np  # noqa: E402

WORKLOADS = {  # name -> (m, n, nnz_per_col, dense_col_nnz)   SURVEY.md 8(d)
    "S2": (100_000, 100_000, 10, 0),
    "S3": (1_000_000, 1_000_000, 8, 0),
    "S5": (1_000_000, 1_000_000, 8, 500_000),
    # not a BASELINE config: S3's sizes with a banded (structured) pattern, to show what the SpMV kernels reach when the
    # gathers share sectors as they do on real LP matrices (VERDICT r1 item 7); reported beside S3, never instead of it
    "S3B": (1_000_000, 1_000_000, 8, 0),
    # ... and with the same 8 offsets in every column (multi-diagonal / stencil-like): a warp's 32 gathers are 32 consecutive
    # doubles, the upper end of sector sharing -- what the kernels reach when the gather pipe is not the limit
    "S3D": (1_000_000, 1_000_000, 8, 0),
}
BANDS = {"S3B": 2048, "S3D": -2048}   # > 0: random rows within the band; < 0: the same offsets in every column (multi-diagonal)
SEED = 12345


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons WHILE the GPU works (B200_PROFILING.md).  NVML is polled from a thread (about
    10 kHz, so that even a 3 ms timed region gets samples); `mark()` brackets the timed region, whose samples are
    reported separately from those of the whole measurement phase (warm-up, timed region, per-kernel timing)."""

    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index=0):
        self.gpu, self.rows, self.marks, self.stop_flag, self.thread, self.err = gpu_index, [], [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].isdigit() else self.gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:   # noqa: BLE001
            self.err = f"NVML unavailable: {e}"[:160]
            return
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def _poll(self):
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:   # noqa: BLE001 -- older bindings
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((time.monotonic(), float(mhz), int(rs)))
            except Exception as e:   # noqa: BLE001
                self.err = str(e)[:160]
                return

    def mark(self):
        self.marks.append(time.monotonic())

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.err or "no samples"], "samples": 0}

        def summary(rows):
            names = sorted(k for k, bit in self.REASONS.items() if any(r[2] & bit for r in rows))
            return {"sm_mhz": float(np.median([r[1] for r in rows])), "min_sm_mhz": float(min(r[1] for r in rows)),
                    "reasons": names, "samples": len(rows)}
        out = summary(self.rows)
        out["sm_max_mhz"] = self.max_mhz
        out["window"] = "warm-up + timed region + per-kernel timing (GPU busy)"
        if len(self.marks) >= 2:
            inside = [r for r in self.rows if self.marks[0] <= r[0] <= self.marks[1]]
            if inside:
                out["timed_region"] = summary(inside)
        return out


def ncu_traffic_bytes(kernel_tag):
    """dram read + write per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/r02_ncu_summary.md, else round 1's; S3 workload); None if the summary is missing"""
    import re
    txt = None
    for name in ("r02_ncu_summary.md", "r01_ncu_summary.md"):
        try:
            txt = open(os.path.join(ROOT, "profiles", name)).read()
            ncu_traffic_bytes.source = f"profiles/{name} (ncu --set full, same kernel, S3)"
            break
        except OSError:
            continue
    if txt is None:
        return None
    for sec in txt.split("\n## ")[1:]:
        if kernel_tag in sec.splitlines()[0]:
            m = re.search(r"traffic = dram read \+ write\*\* \| ([0-9.]+) (\w+)", sec)
            if m:
                return float(m.group(1)) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}.get(m.group(2), 1e6)
    return None


def make_lp(workload):
    from highs_b200.lp import synthetic_lp
    m, n, k, dense = WORKLOADS[workload]
    return synthetic_lp(m, n, k, SEED, dense_col_nnz=dense, band=BANDS.get(workload, 0))


def algorithmic_bytes(n, m, nnz):
    """SURVEY.md 8(d): fp64 values, int32 indices, row pointer / input / output once."""
    b_ax = 12 * nnz + 4 * (m + 1) + 8 * n + 8 * m
    b_aty = 12 * nnz + 4 * (n + 1) + 8 * m + 8 * n
    # fused kernels as built (DESIGN.md "algorithmic bytes"):
    k1 = 8 * 8 * n                 # read x,c,l,u,aty,xSum; write x',xSum
    k2 = b_ax + 6 * 8 * m          # + read y,b,ax,ySum; write y',ySum
    k3 = b_aty + 3 * 8 * n         # + read x,x',aty
    b_iter = b_ax + b_aty + 72 * n + 56 * m   # SURVEY's perfect-fusion iteration model
    return dict(ax=b_ax, aty=b_aty, k1=k1, k2=k2, k3=k3, iter=b_iter)


def reference_rate(lp_path, iters, limit_a=20):
    """steady-state iterations/s of the reference CPU pdlp: two-point fit over two iteration limits"""
    from oracle import binding as ob
    if not ob.ref_available():
        return None
    out = []
    first = None
    for lim in (limit_a, limit_a + iters):
        t = time.monotonic()
        r = ob.run_reference(lp_path=lp_path, options={"pdlp_iteration_limit": lim + 1})
        first = first or r
        out.append((r["pdlp_iteration_count"], r["run_seconds"], time.monotonic() - t))
    (ia, ta, _), (ib, tb, _) = out
    rate = (ib - ia) / max(tb - ta, 1e-9)
    return dict(rate=rate, iters=ib - ia, seconds=tb - ta, setup_seconds=ta - ia / rate, runs=out, first=first)


PARITY_FIELDS = ("objective_function_value", "max_primal_infeasibility", "max_dual_infeasibility", "sum_primal_infeasibilities",
                 "sum_dual_infeasibilities", "max_complementarity_violation", "primal_dual_objective_error")


def parity_block(lp, lp_path, ours, L, ref_run):
    """The north-star parity criterion on THIS workload: after the same L PDHG iterations from the same start, the
    reference's CPU pdlp (oracle/_ref, run through Highs::run()) and this engine return iterates whose objective and
    KKT measures -- both evaluated by the reference's own lpKktCheck (HighsSolution.cpp:1043-1320; ours through
    ref_driver --kkt-of) -- agree to 1e-6 (1 + |ref|).  (Trajectories differ only by the order of the long sums.)"""
    from oracle import binding as ob
    if ours is None or not ob.ref_available():
        return None
    try:
        if ref_run is None:
            ref_run = ob.run_reference(lp_path=lp_path, options={"pdlp_iteration_limit": L + 1})
        mine = ob.reference_kkt(lp, ours, model_status_code=14)   # kIterationLimit
        rows, ok = {}, ours["iters"] == ref_run["pdlp_iteration_count"]
        for k in PARITY_FIELDS:
            if k in ref_run and k in mine:
                a, b = float(mine[k]), float(ref_run[k])
                good = abs(a - b) <= 1e-6 * (1 + abs(b))
                rows[k] = {"ours": a, "reference": b, "ok": bool(good)}
                ok &= good
        return {"iterations": [ours["iters"], ref_run["pdlp_iteration_count"]], "tolerance": "1e-6 * (1 + |reference|)",
                "checked_by": "reference lpKktCheck on both solutions", "fields": rows, "ok": bool(ok)}
    except Exception as e:   # noqa: BLE001 -- the parity block must never break the bench line
        return {"error": str(e)[:300], "ok": False}


def dump_outputs(dirpath, res):
    """What the timed solve returned to its caller -- the four HighsSolution vectors -- as DIR/<name>.npy in float64, so
    that two builds can be compared output for output (the inputs are seeded).  The largest workloads (n = m = 1e6) come
    to 32 MB in all."""
    os.makedirs(dirpath, exist_ok=True)
    for k in ("col_value", "col_dual", "row_value", "row_dual"):
        np.save(os.path.join(dirpath, k + ".npy"), np.asarray(res[k], dtype=np.float64))


def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count()


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    from highs_b200.lp import write_b2lp
    lp = make_lp(args.workload)
    iters = int(min(max(args.steps, 20), 60 if args.workload != "S2" else 400))
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "lp.b2lp")
        write_b2lp(path, lp)
        ref = reference_rate(path, iters)
        hip = None
        if ref is not None:
            # second CPU baseline (SURVEY.md 8(d)): the reference's other first-order engine, solver=hipdlp (40-step blocks)
            try:
                from oracle import binding as ob
                runs = []
                for lim in (40, 40 + 40 * max(1, min(iters, 120) // 40)):
                    r = ob.run_reference(lp_path=path, options={"solver": "hipdlp", "pdlp_iteration_limit": lim})
                    runs.append((r["pdlp_iteration_count"], r["run_seconds"]))
                (ia, ta), (ib, tb) = runs
                hip = {"value": (ib - ia) / max(tb - ta, 1e-9), "unit": "iter/s", "cores": 1, "kind": "reference",
                       "sample": f"HiGHS CPU hipdlp, {ib - ia} steady-state iterations (two-point fit)"}
            except Exception as e:   # noqa: BLE001 -- the extra baseline must never break the line
                hip = {"unavailable": str(e)[:200]}
        tts = None
        if ref is not None and args.to_tolerance > 0:
            from oracle import binding as ob
            t0 = time.monotonic()
            r = ob.run_reference(lp_path=path, options={"kkt_tolerance": args.to_tolerance})
            tts = {"kkt_tolerance": args.to_tolerance, "seconds": time.monotonic() - t0, "run_seconds": r["run_seconds"],
                   "iterations": r["pdlp_iteration_count"], "status": r.get("model_status"),
                   "objective": r.get("objective_function_value")}
    m, n, k, dense = WORKLOADS[args.workload]
    if ref is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_driver missing (build with oracle/build_ref.py)"}))
        return
    line = {
        "impl": "reference", "metric": "pdhg_iterations_per_sec", "value": ref["rate"], "unit": "iter/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / ref["rate"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: synthetic random sparse LP m={m} n={n} nnz={lp.a_matrix_.numNz()} seed={SEED}",
                   "solver": "HiGHS 1.15.1 CPU pdlp (cuPDLP-C), presolve=off, single thread"},
        "cpu_baseline": {"value": ref["rate"], "unit": "iter/s", "cores": 1, "kind": "reference",
                         "host_cores_available": cpu_cores(),
                         "sample": f"{ref['iters']} steady-state iterations (two-point fit over pdlp_iteration_limit, "
                                   f"{ref['seconds']:.1f} s; setup {ref['setup_seconds']:.1f} s excluded)"},
        "e2e": {"value": ref["rate"], "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        # for reading our arm's e2e (which INCLUDES its setup): the reference's own setup and what its end-to-end rate
        # would be for the same number of steps, from the two-point fit (value / e2e above stay the steady-state rate)
        "reference_setup_seconds": ref["setup_seconds"],
        "e2e_same_steps_projection": {"steps": args.steps, "value": args.steps / (ref["setup_seconds"] + args.steps / ref["rate"]),
                                      "unit": "iter/s", "note": "steps / (setup + steps / rate); not measured at this step count"},
        "gpu_launches": 0,
    }
    if tts is not None:
        line["time_to_solution"] = tts
    if hip is not None:
        line["cpu_baseline_hipdlp"] = hip
    print(json.dumps(line))


def run_hipdlp_arm(args, device):
    """HiPDLP mode (SURVEY.md 8(f) rank 2): K Halpern steps (blocks of 40) through b200pdlp_solve_hipdlp on host buffers.
    `value` = steps / CUDA-event time of the device loop (LP resident), `e2e` = steps / wall time of the call."""
    from highs_b200 import engine
    from highs_b200.lp import write_b2lp
    lp = make_lp(args.workload)
    m, n, k, dense = WORKLOADS[args.workload]
    nnz = lp.a_matrix_.numNz()
    K = max(40, (args.steps // 40) * 40)
    W = max(40, (max(args.warmup, 3) + 39) // 40 * 40)
    out_arrays = tuple(np.zeros(q) for q in (n, n, m, m))
    pinned = engine.pin_arrays(engine.lp_arrays(lp) + list(out_arrays))
    sampler = ClockSampler(device)
    sampler.start()
    engine.solve_hipdlp(lp, iter_limit=W, device=device)
    sampler.mark()
    t0 = time.monotonic()
    r = engine.solve_hipdlp(lp, iter_limit=K, device=device)
    wall = time.monotonic() - t0
    sampler.mark()
    clocks = sampler.stop()
    engine.unpin_arrays(pinned)
    assert r["iters"] == K, (r["iters"], K)
    B = algorithmic_bytes(n, m, nnz)
    peak, peak_src = measured_peak_gbs()
    step_bytes = B["ax"] + B["aty"] + 8 * 8 * n + 7 * 8 * m   # 2 SpMV + the x-side (x, xa, c, aty, l, u -> rx, x) and y-side vectors
    value = K / (r["loop_device_ms"] / 1e3)
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import binding as ob
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "lp.b2lp")
            write_b2lp(path, lp)
            runs = []
            for lim in (40, 40 + 40 * (2 if args.workload != "S2" else 10)):
                q = ob.run_reference(lp_path=path, options={"solver": "hipdlp", "pdlp_iteration_limit": lim})
                runs.append((q["pdlp_iteration_count"], q["run_seconds"]))
        (ia, ta), (ib, tb) = runs
        cpu = {"value": (ib - ia) / max(tb - ta, 1e-9), "unit": "iter/s", "cores": 1, "kind": "reference",
               "host_cores_available": cpu_cores(), "sample": f"HiGHS CPU hipdlp, {ib - ia} steady-state steps (two-point fit)"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r)
    print(json.dumps({
        "metric": "pdhg_iterations_per_sec", "value": value, "unit": "iter/s", "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": r["loop_device_ms"] / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: synthetic sparse LP m={m} n={n} nnz={nnz} seed={SEED}",
                   "solver": "hipdlp (reflected Halpern PDHG, blocks of 40 steps, checks between blocks)",
                   "l2": "inputs larger than L2" if args.workload != "S2" else "working set fits L2 (S2)", "parallelism": "single GPU"},
        "gpu_launches": r["kernel_launches"], "wall_seconds": wall, "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": step_bytes * value / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": step_bytes * value / 1e9 / peak, "traffic": None, "kernel": "whole Halpern step (3 launches)",
                     "algorithmic_bytes_per_launch": step_bytes, "peak_source": peak_src},
        "cpu_baseline": cpu,
        "e2e": {"value": K / wall, "unit": "iter/s", "h2d_bytes_per_step": (2 * (12 * nnz + 4 * (n + m)) + 8 * (5 * n + 4 * m)) / K,
                "d2h_bytes_per_step": 8 * (2 * n + 2 * m) / K, "wall_seconds": wall, "setup_seconds": r["setup_seconds"],
                "solve_seconds": r["solve_seconds"]},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--workload", default="S3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity", action="store_true", help="compute the parity block even with --no-cpu-baseline")
    ap.add_argument("--solver", default="pdlp", choices=["pdlp", "hipdlp"],
                    help="pdlp: the cuPDLP-C algorithm (BASELINE's headline, default); hipdlp: the engine's HiPDLP mode "
                         "(reflected Halpern PDHG, solver=hipdlp) against the reference's CPU hipdlp -- single GPU")
    ap.add_argument("--to-tolerance", type=float, default=0.0,
                    help="additionally solve the workload to this kkt_tolerance through the host-buffer call and report the "
                         "wall-clock time to solution (SURVEY.md 8(d)); single GPU / reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the solution vectors the last timed solve returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what this engine computed; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    from highs_b200 import engine
    if engine.device_count() == 0:
        raise SystemExit("bench.py needs a CUDA device; the engine has no CPU fallback")
    if args.solver == "hipdlp":
        if rank == 0:
            run_hipdlp_arm(args, local_rank)
        return
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    lp = make_lp(args.workload)
    m, n, k, dense = WORKLOADS[args.workload]
    nnz = lp.a_matrix_.numNz()
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    prob = engine.Problem(lp, rank=rank, world=world, device=local_rank)
    # B200PDLP_NO_NCCL=1: no NCCL communicator at all -- the fused peer-memory path
    # also assembles the solution (push_rows_kernel); saves the communicator set-up inside the e2e region
    # (default since session D' of round 2; B200PDLP_NO_NCCL=0 brings the communicator back, B200PDLP_NO_P2P=1 needs it)
    no_nccl = os.environ.get("B200PDLP_NO_NCCL", "1") == "1" and os.environ.get("B200PDLP_NO_P2P", "0") != "1"
    if world > 1:
        if not no_nccl:
            ids = [engine.nccl_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            prob.comm_init(ids[0])
        if os.environ.get("B200PDLP_NO_P2P", "0") != "1":
            # fused NVLink path: exchange CUDA-IPC handles of the exchange buffers
            handles = [None] * world
            dist.all_gather_object(handles, prob.p2p_export())
            prob.p2p_import(b"".join(handles))
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- warm-up: W iterations (also captures the CUDA graphs)
    prob.solve(iter_limit=W + 1)
    use_p2p = world > 1 and os.environ.get("B200PDLP_NO_P2P", "0") != "1"
    if use_p2p:
        prob.p2p_timeline()   # reset the device-side timeline
    # ---- timed: exactly K iterations, inputs resident in HBM
    barrier()
    sampler.mark()
    t0 = time.monotonic()
    res = prob.solve(iter_limit=K + 1)
    barrier()
    wall = time.monotonic() - t0
    sampler.mark()
    assert res["iters"] == K, (res["iters"], K)
    timeline = prob.p2p_timeline() if use_p2p else None
    loop_ms = res["loop_device_ms"]
    if dist is not None:
        import torch
        t = torch.tensor([loop_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        loop_ms = float(t.item())
    value = K / (loop_ms / 1e3)
    # ---- per-kernel timing in the real pass sequence (roofline of the dominant kernel)
    reps = 200
    kms = prob.bench_pass(reps)
    B = algorithmic_bytes(prob.n, prob.m, prob.nnz)
    peak, peak_src = measured_peak_gbs()
    k_us = [1e3 * v / reps for v in kms]
    if world == 1:
        dom = 1 if k_us[1] >= k_us[2] else 2
        dom_bytes = B["k2"] if dom == 1 else B["k3"]
        dom_name = "K2 spmv_blocked<Dual> (A x' fused with the dual step)" if dom == 1 else "K3 spmv_blocked<Primal> (A'y' fused with the interaction + step rule)"
    else:
        dom, dom_bytes, dom_name = 1, None, "K2 spmv_blocked<Dual> on the local row block"
    spmv_ms = [prob.bench_spmv(w, 5) and prob.bench_spmv(w, 30) / 30 for w in (0, 1)]
    clocks = sampler.stop() if rank == 0 else None
    # ---- parity: L iterations of this engine (same resident problem, all ranks) for the comparison with the reference
    L_par = 20
    par_sol = None
    if not args.no_cpu_baseline or args.parity:
        par_sol = prob.solve(iter_limit=L_par + 1)
    roofline = None
    if world == 1:
        ach = dom_bytes / (k_us[dom] * 1e-6) / 1e9
        traffic = ncu_traffic_bytes("DualEpilogue" if dom == 1 else "PrimalEpilogue") if args.workload == "S3" else None
        roofline = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                    "traffic_source": getattr(ncu_traffic_bytes, "source", None) if traffic else None,
                    "kernel": dom_name.replace("spmv_blocked", "spmv_sell_kernel"), "algorithmic_bytes_per_launch": dom_bytes, "us_per_launch": k_us[dom],
                    "peak_source": peak_src,
                    "per_kernel_us": {"K1_primal_step": k_us[0], "K2_Ax_dual": k_us[1], "K3_ATy_interaction": k_us[2]},
                    "per_kernel_gbs": {"K1": B["k1"] / k_us[0] / 1e3, "K2": B["k2"] / k_us[1] / 1e3, "K3": B["k3"] / k_us[2] / 1e3},
                    "plain_spmv_gbs": {"Ax": B["ax"] / spmv_ms[0] / 1e6, "ATy": B["aty"] / spmv_ms[1] / 1e6,
                                       "note": "back-to-back launches of one plain SpMV (116 MB) partly hit the 126 MB L2"},
                    "iteration_model": {"bytes": B["iter"], "achieved_gbs": B["iter"] * value / 1e9,
                                        "frac": B["iter"] * value / 1e9 / peak}}
    # ---- e2e: host buffers through the public C-ABI call (single GPU only)
    e2e = None
    tts = None
    if world == 1:
        prob.close()
        # the caller's HighsLp arrays and HighsSolution storage are page-locked once (cudaHostRegister), outside the
        # timed call -- the contract's "inputs in pinned host memory"; B200PDLP_BENCH_PAGEABLE=1 leaves them pageable
        out_arrays = tuple(np.zeros(k) for k in (n, n, m, m))
        pinned = []
        if os.environ.get("B200PDLP_BENCH_PAGEABLE", "0") != "1":
            pinned = engine.pin_arrays(engine.lp_arrays(lp) + list(out_arrays))
        engine.solve(lp, iter_limit=3, device=local_rank, out_arrays=out_arrays)   # untimed: block cache / first-use paths warm
        t0 = time.monotonic()
        r2 = engine.solve(lp, iter_limit=K + 1, device=local_rank, out_arrays=out_arrays)
        e2e_wall = time.monotonic() - t0
        a = lp.a_matrix_
        dev_prep = os.environ.get("B200PDLP_DEVICE_PREP", "1") != "0"
        # device prologue: the HighsLp arrays go up once (CSC + 3 n-vectors + 2 m-vectors); host prologue: both layouts + vectors
        h2d = (12 * nnz + 4 * (n + 1) + 24 * n + 16 * m) if dev_prep else (2 * (12 * nnz + 4 * (n + m)) + 8 * (5 * n + 3 * m))
        d2h = 8 * (2 * n + 2 * m)
        e2e = {"value": K / e2e_wall, "unit": "iter/s", "h2d_bytes_per_step": h2d / K, "d2h_bytes_per_step": d2h / K,
               "wall_seconds": e2e_wall, "setup_seconds": r2["setup_seconds"], "solve_seconds": r2["solve_seconds"],
               "host_buffers": "page-locked (cudaHostRegister, outside the timed call)" if pinned else "pageable",
               "note": "one b200pdlp_solve call on host buffers: H2D of the HighsLp arrays, prologue (formulate + scaling + "
                       "transposition + layouts"
                       + (" on the device" if dev_prep else " on host threads") + "), K iterations, postsolve, D2H of the "
                       "HighsSolution; bytes are per call divided by K; measured on the second call of the process (one untimed "
                       "3-iteration call first: the library's device-block cache and CUDA module are warm, as in any process that "
                       "solves more than one LP)"}
        if args.to_tolerance > 0:
            tol = args.to_tolerance
            t0 = time.monotonic()
            r3 = engine.solve(lp, tol_primal=tol, tol_dual=tol, tol_gap=tol, iter_limit=2_000_000, device=local_rank,
                              out_arrays=out_arrays)
            tts = {"kkt_tolerance": tol, "seconds": time.monotonic() - t0, "iterations": r3["iters"], "status": r3["term_name"],
                   "objective": lp.objectiveValue(r3["col_value"]), "setup_seconds": r3["setup_seconds"],
                   "solve_seconds": r3["solve_seconds"]}
        if pinned:
            engine.unpin_arrays(pinned)
    else:
        # N > 1: host buffers -> row/column shards on every GPU (formulate+scale on every rank, layouts, H2D),
        # communicator + peer-memory setup, K iterations, assembled HighsSolution back on the host
        import torch
        if use_p2p:
            prob.p2p_release()
        barrier()
        prob.close()
        barrier()
        t0 = time.monotonic()
        prob2 = engine.Problem(lp, rank=rank, world=world, device=local_rank)
        if not no_nccl:
            ids = [engine.nccl_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            prob2.comm_init(ids[0])
        if use_p2p:
            handles = [None] * world
            dist.all_gather_object(handles, prob2.p2p_export())
            prob2.p2p_import(b"".join(handles))
        r2 = prob2.solve(iter_limit=K + 1)
        barrier()
        e2e_wall = time.monotonic() - t0
        t = torch.tensor([e2e_wall], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_wall = float(t.item())
        h2d = (2 * (12 * nnz + 4 * (n + m)) + 8 * (5 * n + 3 * m)) / world
        e2e = {"value": K / e2e_wall, "unit": "iter/s", "h2d_bytes_per_step": h2d / K, "d2h_bytes_per_step": 8 * (2 * n + 2 * m) / K,
               "wall_seconds": e2e_wall, "solve_seconds": r2["solve_seconds"],
               "note": "per rank: Problem create (formulate + scale on the rank's GPU unless B200PDLP_MG_DEVICE_PREP=0, its layouts on "
                       "the host, H2D of its shard), " + ("" if no_nccl else "NCCL communicator + ")
                       + "CUDA-IPC peer mapping, K iterations, gather + D2H of the solution; max over ranks"}
        if use_p2p:
            prob2.p2p_release()
        barrier()
        prob2.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    # ---- CPU baseline: the reference itself on this box's host cores (bounded sample)
    cpu = None
    parity = None
    if not args.no_cpu_baseline or args.parity:
        from highs_b200.lp import write_b2lp
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "lp.b2lp")
            write_b2lp(path, lp)
            ref = reference_rate(path, 40 if args.workload != "S2" else 400, limit_a=L_par) if not args.no_cpu_baseline else None
            parity = parity_block(lp, path, par_sol, L_par, ref["first"] if ref else None)
        if ref:
            cpu = {"value": ref["rate"], "unit": "iter/s", "cores": 1, "kind": "reference",
                   "host_cores_available": cpu_cores(),
                   "sample": f"{ref['iters']} steady-state iterations of HiGHS CPU pdlp on the same LP (two-point fit, "
                             f"{ref['seconds']:.1f} s; O(nnz) setup of {ref['setup_seconds']:.1f} s excluded)"}
    line = {
        "metric": "pdhg_iterations_per_sec", "value": value, "unit": "iter/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": loop_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: synthetic random sparse LP m={m} n={n} nnz={nnz} seed={SEED}"
                               + (f" + one column with {dense} nonzeros" if dense else "")
                               + (f" -- BANDED pattern (rows within {BANDS[args.workload]} of the diagonal; structured, "
                                  "not a BASELINE config)" if BANDS.get(args.workload, 0) > 0 else "")
                               + (f" -- MULTI-DIAGONAL pattern (the same offsets within {-BANDS[args.workload]} of the diagonal in "
                                  "every column; structured, not a BASELINE config)" if BANDS.get(args.workload, 0) < 0 else ""),
                   "options": "solver=pdlp presolve=off, adaptive step + restarts, checks every 40 iterations",
                   "l2": "inputs larger than L2 (one iteration streams ~0.37 GB vs 126 MB L2)" if args.workload != "S2"
                         else "working set fits L2 (S2)",
                   "parallelism": (f"row blocks + column shards x{world}, "
                                   + ("reduce-scatter/all-gather fused into our kernels over NVLink peer memory"
                                      if os.environ.get("B200PDLP_NO_P2P", "0") != "1" else "NCCL reduce-scatter + all-gather"))
                   if world > 1 else "single GPU"},
        "gpu_launches": res["kernel_launches"], "passes": res["passes"], "restarts": res["restarts"],
        "wall_seconds": wall, "pass_device_ms": res["iter_device_ms"],
        "phase_us": (None if world == 1 else {"primal_shard+allgather": k_us[0], "Ax+dual": k_us[1], "partial_ATy": k_us[2],
                                              "reduce_scatter+step_rule": k_us[3]}),
        "p2p_timeline_us": timeline, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
        "parity": parity,
    }
    if tts is not None:
        line["time_to_solution"] = tts
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
