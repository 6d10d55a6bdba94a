#!/usr/bin/env python
"""Benchmark of the BP5 hot path (driver contract: one JSON line on stdout).

    python bench.py --gpus N --steps K --warmup W            # our arm (B200)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also write the last timed solve's outputs

Metric (BASELINE.json / bp5/step-64.cu:458-461): DoFs x CG iterations / second,
as the reference's "pcg-merged" block measures it: one STEP is one full merged
CG solve `IterationNumberControl(200, 1e-6*|b|)` of the BP5 Poisson problem,
x0 = 0, b = int phi_i, including the x = 0 reset (bp5/step-64.cu:481-517).

Workload at N=1: BP5, p = 6, 88^3 cells = 529^3 = 148,035,889 DoFs, fp64 --
config 4's per-GPU block (SURVEY.md 8d), the largest single-GPU configuration;
every vector (1.18 GB) and the metric (11.2 GB) are far larger than the 126 MB
L2, so no L2 flush is needed between steps.  Headline quadrature: Gauss-Lobatto
collocation (north star); the reference's shipped default QGauss(p+1)
(bp5/step-64.cu:246, COLLOCATION commented out) is measured in the same run and
reported under "variants".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "BP5 merged-CG throughput (DoFs x CG iterations per second)"
UNIT = "GDoF*it/s"
MAX_ITS = 200


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--degree", type=int, default=6)
    ap.add_argument("--cells", type=int, default=88, help="cells per direction per GPU")
    ap.add_argument("--quadrature", default="gll", choices=["gll", "gauss"])
    ap.add_argument("--transport", default="peer", choices=["peer", "nccl"],
                    help="N>1: halo + scalar exchange through peer memory (library kernels) or NCCL")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N>1: weak = --cells^3 cells per GPU; strong = --cells^3 cells in total, split over the GPUs")
    ap.add_argument("--geometry", default="stored", choices=["stored", "otf"],
                    help="stored metric tensor (headline) or geometry recomputed in the kernel (config 5; gll only)")
    ap.add_argument("--deformation", type=float, default=0.0, help="eps of the smooth mesh deformation (config 5: 0.1)")
    ap.add_argument("--no-variants", action="store_true", help="skip the second quadrature")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-cells", type=int, default=0, help="cells per direction of the CPU sample (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed solve of each quadrature returned as DIR/<quadrature>_x.npy (a "
                         "seeded sample of the solution) and DIR/<quadrature>_solve.npy (iterations, final residual, "
                         "|x|_2), so that two builds can be compared output for output (one GPU only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    return args


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- CPU arm
def cpu_arm(degree, quad_name, cells, iterations, repeats=1):
    """Times the oracle's merged CG (CPU restatement of the reference's deal.II path; the
    reference itself needs deal.II+MPI+p4est and cannot be built here) on the host cores."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle as O
    quad = O.GLL if quad_name == "gll" else O.GAUSS
    # all host cores, whatever OMP_NUM_THREADS says: torchrun exports OMP_NUM_THREADS=1 to every rank, which made
    # the N>1 reference runs of round 1 single-threaded (cores differed between N=1 and N>1)
    O.lib().orc_set_num_threads(host_threads())
    m = O.OracleMesh(degree, (cells,) * 3, quad=quad)
    b = m.rhs()
    best = None
    # timing only: the vectorisable collocation cell operator for GLL (same results to 1e-16, tests pin it);
    # Gauss quadrature runs the general evaluator
    O.lib().orc_set_fast_path(1)
    try:
        for _ in range(repeats):
            t0 = time.perf_counter()
            x, its, res, hist, ok = m.cg(b, variant=1, control=0, tol=0.0, max_its=iterations)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    finally:
        O.lib().orc_set_fast_path(0)
    return {"value": m.n_dofs * its / best / 1e9, "unit": UNIT, "cores": O.lib().orc_num_threads(),
            "kind": "port", "seconds": best,
            "sample": f"BP5 p={degree} {quad_name}, {cells}^3 cells = {m.n_dofs} DoFs, {its} merged-CG iterations "
                      f"(OpenMP oracle, restatement of the deal.II CPU path, not deal.II itself"
                      f"{'; vectorisable collocation cell operator' if quad_name == 'gll' else ''})"}, m.n_dofs


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def auto_cpu_cells(degree):
    # ~1M DoFs: a few seconds per 10 iterations on 8-64 cores
    return max(4, round((1.0e6 ** (1 / 3) - 1) / degree))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cells = args.cpu_cells or auto_cpu_cells(args.degree)
    iters = 10
    t_all = time.perf_counter()
    vals = []
    for _ in range(args.warmup):
        cpu_arm(args.degree, args.quadrature, cells, 2)
        if time.perf_counter() - t_all > 60:
            break
    ms = []
    for _ in range(args.steps):
        r, ndofs = cpu_arm(args.degree, args.quadrature, cells, iters)
        vals.append(r)
        ms.append(r["seconds"] * 1e3)
    tot_s = sum(v["seconds"] for v in vals)
    value = ndofs * iters * len(vals) / tot_s / 1e9
    cb = dict(vals[0]); cb["value"] = value; cb.pop("seconds", None)
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": sum(ms) / len(ms), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": f"BP5 p={args.degree} {args.quadrature}, bounded CPU sample {cells}^3 cells, "
                                  f"{iters} merged-CG iterations per step",
                      "full_workload": f"BP5 p={args.degree}, {args.cells}^3 cells per GPU, {MAX_ITS} iterations"},
           "cpu_baseline": cb, "gpu_launches": 0,
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))
    return 0


# --------------------------------------------------------------------------- GPU arm
DUMP_SAMPLE = 1 << 21          # solution entries --dump-outputs writes per quadrature: 16 MB in fp64


def solution_sample(x):
    """the whole vector if it is small, else its entries at DUMP_SAMPLE indices drawn with a fixed seed: the same
    indices for the same mesh on every run and every build"""
    import numpy as np
    if x.size <= DUMP_SAMPLE:
        return x
    return x[np.sort(np.random.default_rng(0).choice(x.size, DUMP_SAMPLE, replace=False))]


def measure_solver(dc, torch, ctx, stream, op, steps, warmup, sampler=None, dump=False):
    """K timed merged-CG solves, device-resident b; returns dict of results.  dump: also return what the caller of
    the last timed solve received (under "outputs")."""
    import numpy as np
    n = op.n_owned
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    bnorm = b.l2_norm()
    control = dc.IterationNumberControl(MAX_ITS, 1e-6 * bnorm)
    solver = dc.SolverCGFullMerge(control)
    op.do_zero_out = False          # bp5/step-64.cu:483
    for _ in range(warmup):
        x.set(0.0)
        solver.solve(op, x, b, history=False)
    ctx.synchronize()
    launches0 = ctx.launch_count
    # the timed loop runs the path users get: CUDA-graph replay of the iteration batches, no per-launch events
    # (bp5_operator_profile switches the graph off -- that is the separate short pass below)
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    its_total = 0
    for _ in range(steps):
        x.set(0.0)                  # solution_dev = 0, bp5/step-64.cu:491 (inside the timer)
        solver.solve(op, x, b, history=False)
        its_total += control.last_step()
    e1.record(stream)
    e1.synchronize()
    secs = e0.elapsed_time(e1) * 1e-3
    launches = ctx.launch_count - launches0
    xnorm = x.l2_norm()
    last_value = control.last_value()
    outputs = None
    if dump:
        # taken here: the profiled pass below solves into the same x
        outputs = {"x": solution_sample(x.to_host()),
                   "solve": np.array([control.last_step(), last_value, xnorm], dtype=np.float64)}
    # profiled pass, still under the clock sampler: the same solve with a CUDA event pair around every launch of
    # the dominant kernel (graph replay off), for roofline.achieved; also timed as a whole for comparison
    op.profile(True)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    prof_its = 0
    for _ in range(max(1, min(2, steps))):
        x.set(0.0)
        solver.solve(op, x, b, history=False)
        prof_its += control.last_step()
    p1.record(stream)
    p1.synchronize()
    prof_secs = p0.elapsed_time(p1) * 1e-3
    k_launches, k_ms = op.profile_result()
    op.profile(False)
    clocks = sampler.stop() if sampler else None
    res = dict(secs=secs, its_total=its_total, its_per_step=its_total / steps, n=n, launches=launches,
               kernel_launches=k_launches, kernel_ms=k_ms, bnorm=bnorm, xnorm=xnorm, last_value=last_value,
               clocks=clocks, prof_secs=prof_secs, prof_its=prof_its, outputs=outputs)
    b.close(); x.close()
    return res


def measure_e2e(dc, torch, ctx, stream, op, steps, warmup):
    """Same solve through the host-buffer entry point: pinned host b / x0 in, x out, copies timed."""
    import numpy as np
    n = op.n_owned
    b = op.initialize_dof_vector()
    op.assemble_rhs(b)
    bh = torch.empty(n, dtype=torch.float64, pin_memory=True)
    xh = torch.empty(n, dtype=torch.float64, pin_memory=True)
    bh.numpy()[:] = b.to_host()
    bnorm = float(np.linalg.norm(bh.numpy()))
    b.close()
    control = dc.IterationNumberControl(MAX_ITS, 1e-6 * bnorm)
    op.do_zero_out = False
    xnp, bnp = xh.numpy(), bh.numpy()
    for _ in range(max(1, min(warmup, 1))):
        dc.cg_solve_host(op, xnp, bnp, control, x0_is_zero=True)
    t0 = time.perf_counter()
    its_total = 0
    for _ in range(steps):
        # zero initial guess like the reference driver (bp5/step-64.cu:491): H2D b; solve; D2H x; returns after the copy back
        dc.cg_solve_host(op, xnp, bnp, control, x0_is_zero=True)
        its_total += control.last_step()
    secs = time.perf_counter() - t0
    return dict(secs=secs, its_total=its_total, h2d=n * 8, d2h=n * 8, xnorm=float(np.linalg.norm(xnp)))


def measure_helmholtz(dc, torch, ctx, stream):
    """BASELINE configs[1]: step-64 variable-coefficient Helmholtz, p=4, 64^3 cells = 257^3 DoFs, merged CG with
    SolverControl(n_dofs, 1e-12|b|) (step-64/step-64.cu:513-514).  Reported under "variants"; never fatal."""
    try:
        op = dc.PoissonOperator(ctx, dc.make_problem(4, (64, 64, 64), operator_kind=dc.OP_HELMHOLTZ, upper=(1., 1., 1.)))
        b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
        op.assemble_rhs(b)
        n = op.n_owned
        op.do_zero_out = False
        control = dc.SolverControl(n, 1e-12 * b.l2_norm())
        secs = None
        for rep in range(2):                      # warm-up, then timed
            x.set(0.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            dc.SolverCGFullMerge(control).solve(op, x, b, history=False)
            e1.record(stream)
            e1.synchronize()
            secs = e0.elapsed_time(e1) * 1e-3
        out = {"workload": "step-64 Helmholtz, p=4, 64^3 cells, SolverControl(n_dofs, 1e-12|b|), QGauss(5)", "dofs": n,
               "iterations": control.last_step(), "value": n * control.last_step() / secs / 1e9, "unit": UNIT,
               "ms_per_solve": secs * 1e3, "kernel": op.kernel_name, "solution_norm_L2": op.l2_norm(x)}
        b.close(); x.close(); op.close()
        return out
    except Exception as e:                        # a side measurement must not cost the headline line
        return {"error": f"{type(e).__name__}: {e}"}


def measure_affine_otf(dc, torch, ctx, stream, args, hbm_peak):
    """Geometry on the fly on the headline's (undeformed) mesh: no metric stream at all, the kernel forms
    G = w_q diag(hy hz / hx, ...) from three constants (bp5_problem_t.geometry_mode = BP5_GEOM_ON_THE_FLY, affine fast
    path).  The headline stays on the stored metric tensor (north star, general meshes); this variant shows what
    recomputation buys where it is cheap.  Reported under "variants"; never fatal."""
    try:
        op = dc.PoissonOperator(ctx, dc.make_problem(args.degree, (args.cells,) * 3, quadrature=dc.QUAD_GLL,
                                                     geometry_mode=dc.GEOM_ON_THE_FLY))
        r = measure_solver(dc, torch, ctx, stream, op, max(1, min(args.steps, 2)), 1)
        bytes_vmult, bytes_cg = op.algorithmic_bytes()
        k_s = r["kernel_ms"] * 1e-3 / max(1, r["kernel_launches"])
        out = {"workload": f"BP5 p={args.degree} GLL, {args.cells}^3 cells, geometry on the fly (affine fast path), merged CG",
               "kernel": op.kernel_name, "value": r["n"] * r["its_total"] / r["secs"] / 1e9, "unit": UNIT,
               "ms_per_step": r["secs"] / max(1, min(args.steps, 2)) * 1e3, "cell_kernel_ms": k_s * 1e3,
               "cell_kernel_gdofs": r["n"] / k_s / 1e9, "algorithmic_bytes_per_launch": bytes_vmult,
               "cell_kernel_frac_of_hbm": bytes_vmult / k_s / 1e9 / hbm_peak,
               "note": "16 B/DoF: this kernel is bound by the shared-memory pipe and fp64 issue, not by HBM", "x_l2": r["xnorm"]}
        op.close()
        return out
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def measure_config5_otf(dc, torch, ctx, stream):
    """BASELINE config 5 (stored metric tensor vs geometry on the fly) on a smoothly deformed mesh with the reference's
    default quadrature QGauss(p+1): p = 5, 60^3 cells, 200 merged-CG iterations in both geometry modes.  The
    on-the-fly kernel (apply_otfg.cuh) rebuilds the coefficient from the nodal coordinates: a quarter of the geometry
    bytes at about half the rate.  Reported under "variants"; never fatal."""
    try:
        out = {"workload": "BP5 p=5 QGauss(6), 60^3 cells deformed (eps 0.1) = 27270901 DoFs, 200 merged-CG iterations"}
        for mode, key in ((dc.GEOM_STORED, "stored_metric"), (dc.GEOM_ON_THE_FLY, "on_the_fly")):
            op = dc.PoissonOperator(ctx, dc.make_problem(5, (60, 60, 60), deformation=1, eps=0.1, geometry_mode=mode))
            b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
            op.assemble_rhs(b)
            control = dc.IterationNumberControl(MAX_ITS, 1e-6 * b.l2_norm())
            op.do_zero_out = False
            solver = dc.SolverCGFullMerge(control)
            x.set(0.0); solver.solve(op, x, b, history=False)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            x.set(0.0)
            e0.record(stream); solver.solve(op, x, b, history=False); e1.record(stream); e1.synchronize()
            secs = e0.elapsed_time(e1) * 1e-3
            out[key] = {"kernel": op.kernel_name, "value": op.n_owned * control.last_step() / secs / 1e9, "unit": UNIT,
                        "iterations": control.last_step(), "last_residual": control.last_value(), "x_l2": x.l2_norm(),
                        "geometry_bytes": op.algorithmic_bytes()[0] - 16.0 * op.n_owned}
            b.close(); x.close(); op.close()
        out["on_the_fly_over_stored"] = out["on_the_fly"]["value"] / out["stored_metric"]["value"]
        return out
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def measure_small_mesh(dc, torch, ctx, stream, args):
    """The N=1 point of the small strong-scaling mesh of the N>1 lines (bench_multi.py `strong_small_mesh`:
    (cells/2)^3 cells split over the GPUs): the same mesh on one GPU, so that a strong-scaling efficiency can be formed
    from driver-run numbers alone.  Reported under "variants"; never fatal."""
    try:
        cells = max(8, args.cells // 2)
        op = dc.PoissonOperator(ctx, dc.make_problem(args.degree, (cells,) * 3, quadrature=dc.QUAD_GLL))
        b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
        op.assemble_rhs(b)
        control = dc.IterationNumberControl(MAX_ITS, 1e-6 * b.l2_norm())
        op.do_zero_out = False
        solver = dc.SolverCGFullMerge(control)
        for _ in range(2):
            x.set(0.0); solver.solve(op, x, b, history=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        its = 0
        for _ in range(3):
            x.set(0.0); solver.solve(op, x, b, history=False)
            its += control.last_step()
        e1.record(stream); e1.synchronize()
        secs = e0.elapsed_time(e1) * 1e-3
        out = {"workload": f"BP5 p={args.degree} GLL, {cells}^3 cells = {op.n_owned} DoFs on one GPU (N=1 point of the N>1 "
                           f"lines' strong_small_mesh)", "dofs": op.n_owned, "value": op.n_owned * its / secs / 1e9, "unit": UNIT,
               "ms_per_iteration": secs / max(1, its) * 1e3, "x_l2": x.l2_norm()}
        b.close(); x.close(); op.close()
        return out
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def measure_refined_mesh(dc, torch, ctx, stream, args):
    """Merged CG through the tuned kernel on a locally refined mesh (hanging nodes on the faces of the refined box,
    the `constraint_mask` slot of bp5/fe_evaluation_gl.h:88,150,167): (cells/2)^3 coarse cells, the corner octant refined
    once.  Reported under "variants"; never fatal."""
    try:
        cells = max(8, args.cells // 2)
        op = dc.PoissonOperator(ctx, dc.make_problem(args.degree, (cells,) * 3, quadrature=dc.QUAD_GLL, refine_lo=(0, 0, 0),
                                                     refine_hi=(cells // 2,) * 3))
        b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
        op.assemble_rhs(b)
        control = dc.IterationNumberControl(MAX_ITS, 1e-6 * b.l2_norm())
        op.do_zero_out = False
        solver = dc.SolverCGFullMerge(control)
        x.set(0.0); solver.solve(op, x, b, history=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        x.set(0.0); solver.solve(op, x, b, history=False)
        its = control.last_step()
        e1.record(stream); e1.synchronize()
        secs = e0.elapsed_time(e1) * 1e-3
        out = {"workload": f"BP5 p={args.degree} GLL, {cells}^3 coarse cells with the corner {cells // 2}^3 refined once = "
                           f"{op.n_cells} cells, {op.n_owned} DoFs (hanging nodes), merged CG, tuned kernel",
               "dofs": op.n_owned, "cells": op.n_cells, "value": op.n_owned * its / secs / 1e9, "unit": UNIT,
               "ms_per_iteration": secs / max(1, its) * 1e3, "x_l2": x.l2_norm()}
        b.close(); x.close(); op.close()
        return out
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def measure_user_functor(hbm_peak):
    """What staying on the reference's device-functor API costs (examples/bp5_functors.cu bench mode): the user-written
    LocalPoissonOperator on CUDAWrappers::MatrixFree / FEEvaluationGL (one CTA per cell, deal.II-layout arrays) against
    the tuned kernel, p = 6 GLL, 42^3 cells = 16.2 M DoFs.  Reported under "variants"; never fatal."""
    exe = os.path.join(ROOT, "build", "examples", "bp5_functors")
    try:
        if not os.path.exists(exe):
            return {"error": "build/examples/bp5_functors not built"}
        out = subprocess.run([exe, "bench", "6", "42"], capture_output=True, text=True, timeout=300)
        d = json.loads(out.stdout.strip().splitlines()[-1])
        ach = d["algorithmic_bytes_per_vmult"] / (d["user_functor_vmult_ms"] * 1e-3) / 1e9
        ach_lib = d["algorithmic_bytes_per_vmult"] / (d["library_vmult_ms"] * 1e-3) / 1e9
        return {"workload": f"BP5 vmult through user-written device functors, p=6 GLL, {d['cells']}^3 cells = {d['dofs']} DoFs",
                "vmult_ms": d["user_functor_vmult_ms"], "value": d["dofs"] / (d["user_functor_vmult_ms"] * 1e-3) / 1e9,
                "unit": "GDoF/s", "roofline_achieved": ach, "roofline_frac": ach / hbm_peak,
                "tuned_kernel_vmult_ms": d["library_vmult_ms"], "tuned_kernel_roofline_frac": ach_lib / hbm_peak,
                "rel_diff_vs_tuned_kernel": d["rel_diff"]}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def run_b200(args):
    import numpy as np
    import torch
    import dealceed_b200 as dc

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one rank per GPU)")
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs: one GPU only")
        import bench_multi
        return bench_multi.run(args)

    torch.cuda.set_device(local_rank)
    ctx = dc.Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    quad_ids = {"gll": dc.QUAD_GLL, "gauss": dc.QUAD_GAUSS}
    order = [args.quadrature] + ([] if args.no_variants else [q for q in ("gll", "gauss") if q != args.quadrature])
    results = {}
    for qi, qname in enumerate(order):
        geom = dc.GEOM_ON_THE_FLY if args.geometry == "otf" else dc.GEOM_STORED
        op = dc.PoissonOperator(ctx, dc.make_problem(args.degree, (args.cells,) * 3, quadrature=quad_ids[qname],
                                                     deformation=1 if args.deformation else 0, eps=args.deformation,
                                                     geometry_mode=geom))
        sampler = ClockSampler(local_rank) if qi == 0 else None
        r = measure_solver(dc, torch, ctx, stream, op, args.steps, args.warmup, sampler, dump=bool(args.dump_outputs))
        bytes_vmult, bytes_cg = op.algorithmic_bytes()
        r["bytes_vmult"], r["bytes_cg"], r["kernel"] = bytes_vmult, bytes_cg, op.kernel_name
        if qi == 0:
            r["e2e"] = measure_e2e(dc, torch, ctx, stream, op, max(1, min(args.steps, 3)), args.warmup)
        results[qname] = r
        op.close()
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for qname, r in results.items():
            for name, a in r.pop("outputs").items():
                np.save(os.path.join(args.dump_outputs, f"{qname}_{name}.npy"), a)
    helm = affine = small = refined = config5 = None
    if not args.no_variants:
        helm = measure_helmholtz(dc, torch, ctx, stream)
        config5 = measure_config5_otf(dc, torch, ctx, stream)
        small = measure_small_mesh(dc, torch, ctx, stream, args)
        refined = measure_refined_mesh(dc, torch, ctx, stream, args)
        if not args.deformation:
            affine = measure_affine_otf(dc, torch, ctx, stream, args, hbm_peak)
    ctx.close()

    def summarize(r):
        value = r["n"] * r["its_total"] / r["secs"] / 1e9
        k_s = r["kernel_ms"] * 1e-3 / max(1, r["kernel_launches"])
        ach = r["bytes_vmult"] / k_s / 1e9
        return value, ach, k_s

    def cg_fracs(r):
        # whole iteration against the byte models of SURVEY 8(d): 72 + 48 r per DoF (the contract figure, diagonal
        # counted) and 64 + 48 r (the all-ones diagonal is recognised and never read: the honest denominator)
        rate = r["its_total"] / r["secs"] / 1e9
        return r["bytes_cg"] * rate / hbm_peak, (r["bytes_cg"] - 8.0 * r["n"]) * rate / hbm_peak

    head = results[args.quadrature]
    value, ach, k_s = summarize(head)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(f"p{args.degree}_{args.quadrature}_{args.cells}")
        except Exception:
            traffic = None
    e2e = head["e2e"]
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": head["secs"] / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": f"BP5 Poisson, p={args.degree}, {args.cells}^3 cells = {head['n']} DoFs on one B200, "
                        f"{args.quadrature} quadrature (p+1 points), merged CG, IterationNumberControl({MAX_ITS}, 1e-6|b|), "
                        f"{head['its_per_step']:.0f} iterations per step",
            "quadrature": args.quadrature, "degree": args.degree, "cells_per_gpu": args.cells ** 3,
            "geometry": "on-the-fly" if args.geometry == "otf" else "stored metric tensor", "deformation_eps": args.deformation,
            "dofs_per_gpu": head["n"], "parallelism": "1 block", "iterations_per_step": head["its_per_step"],
            "l2": "no flush: every vector (8 B x DoFs) and the metric are larger than the 126 MB L2",
            "kernel": head["kernel"],
        },
        "clocks": head["clocks"],
        "e2e": {"value": head["n"] * e2e["its_total"] / e2e["secs"] / 1e9, "unit": UNIT,
                "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                "api": "bp5_cg_solve_host (pinned host b -> device, zero initial guess, solve, x -> pinned host)"},
        "gpu_launches": head["launches"],
        "roofline": {
            "bound": "hbm", "kernel": head["kernel"], "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
            "frac": ach / hbm_peak, "frac_of_nominal_8000": ach / 8000.0, "peak_source": peak_src,
            "traffic": traffic, "algorithmic_bytes_per_launch": head["bytes_vmult"],
            "avg_launch_ms": k_s * 1e3, "launches_timed": head["kernel_launches"],
            "kernel_share_of_step": head["kernel_ms"] * 1e-3 / head["prof_secs"],
            "timing": "value / ms_per_step: the shipped path (CUDA-graph replay of the iteration batches); "
                      "avg_launch_ms: CUDA events around every launch of the cell kernel in a separate profiled pass "
                      "of the same solve (graph replay off), whose whole-solve rate is profiled_pass_value",
            "profiled_pass_value": head["n"] * head["prof_its"] / head["prof_secs"] / 1e9,
            "cg_achieved": head["bytes_cg"] * head["its_total"] / head["secs"] / 1e9,
            "cg_frac": cg_fracs(head)[0], "cg_frac_64B_model": cg_fracs(head)[1],
        },
        "check": {"x_l2": head["xnorm"], "b_l2": head["bnorm"], "last_residual": head["last_value"],
                  "e2e_x_l2": e2e["xnorm"]},
    }
    variants = {}
    for qname, r in results.items():
        if qname == args.quadrature:
            continue
        v, a, ks = summarize(r)
        variants[qname] = {"value": v, "unit": UNIT, "ms_per_step": r["secs"] / args.steps * 1e3,
                           "kernel": r["kernel"], "roofline_achieved": a, "roofline_frac": a / hbm_peak,
                           "avg_launch_ms": ks * 1e3, "iterations_per_step": r["its_per_step"],
                           "cg_frac": cg_fracs(r)[0], "cg_frac_64B_model": cg_fracs(r)[1], "x_l2": r["xnorm"]}
    if helm is not None:
        variants["helmholtz_config2"] = helm
    if affine is not None:
        variants["geometry_on_the_fly_affine"] = affine
    if small is not None:
        variants["strong_small_mesh_n1"] = small
    if refined is not None:
        variants["locally_refined_mesh"] = refined
    if not args.no_variants:
        variants["user_functor"] = measure_user_functor(hbm_peak)
        if config5 is not None:
            variants["config5_geometry_on_the_fly"] = config5
    out["variants"] = variants
    if not args.no_cpu_baseline:
        cells = args.cpu_cells or auto_cpu_cells(args.degree)
        cb, _ = cpu_arm(args.degree, args.quadrature, cells, 10)
        cb.pop("seconds", None)
        out["cpu_baseline"] = cb
    print(json.dumps(out))
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
