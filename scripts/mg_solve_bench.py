"""Time to solution of the multigrid-preconditioned CG against plain and Jacobi CG, and the parts of one V-cycle.

For each mesh (default: p = 6 GLL on 88^3 cells, levels 88/44/22/11, and on 96^3 cells, levels down to 3^3):
  * iterations and device-synchronised wall time to 1e-8 |b| of: merged CG without preconditioner, merged CG with
    Jacobi, and standard CG with the multigrid V-cycle (set-up time reported separately);
  * one V-cycle split by CUDA events into operator applications per level, transfers, Chebyshev / residual vector
    kernels and the coarse solve (bp5_mg_profile), averaged over --vcycles V-cycles;
  * the transfer kernels' algorithmic bytes per second (prolongation and restriction per level, timed alone)
    against the copy peak measured for DESIGN.md section 3.3 (6548.2 GB/s);
  * the card name, power limit and SM clock, read in the same run.
Writes one JSON document to --out (and stdout).

    python scripts/mg_solve_bench.py --out profiles/mg_solve_bench_b200.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_PEAK_GBS = 6548.2     # DESIGN.md section 3.3, measured copy rate of the B200 the library was tuned on


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    first = out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else ""
    return dict(zip(q.split(","), [v.strip() for v in first.split(",")])) if first else {"error": out.stderr.strip()}


def timed(ctx, fn, reps=1):
    ctx.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    ctx.synchronize()
    return (time.perf_counter() - t0) / reps


def run_mesh(dc, ctx, p, cells, tol_rel, max_its, n_vcycles):
    op = dc.PoissonOperator(ctx, dc.make_problem(p, (cells,) * 3, quadrature=dc.QUAD_GLL))
    b, x, diag = op.initialize_dof_vector(), op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    tol = tol_rel * b.l2_norm()
    op.compute_diagonal(diag, invert=True)
    res = dict(degree=p, cells=cells, dofs=op.n_owned, tol_rel=tol_rel)

    def solve(kind, mg=None):
        ctl = dc.SolverControl(max_its, tol)
        x.set(0.0)
        op.do_zero_out = kind != "merged"
        if kind == "merged":
            f = lambda: dc.SolverCGFullMerge(ctl).solve(op, x, b, history=False)
        elif kind == "jacobi":
            f = lambda: dc.SolverCGFullMerge(ctl).solve(op, x, b, preconditioner=diag, history=False)
        else:
            f = lambda: dc.SolverCG(ctl).solve(op, x, b, preconditioner=mg, history=False)
        t = timed(ctx, f)
        return dict(iterations=ctl.last_step(), seconds=t, l2_norm=op.l2_norm(x))

    # warm-up of every path (module load, graph capture) on a short solve, then the timed solves
    for kind in ("merged", "jacobi"):
        ctl = dc.SolverControl(30, 0.0)
        x.set(0.0)
        try:
            (dc.SolverCGFullMerge(ctl).solve(op, x, b, preconditioner=diag if kind == "jacobi" else None))
        except dc.NoConvergence:
            pass
    res["plain_merged_cg"] = solve("merged")
    res["jacobi_merged_cg"] = solve("jacobi")
    ctx.synchronize()
    t0 = time.perf_counter()
    mg = dc.Multigrid(op)
    ctx.synchronize()
    res["mg_setup_seconds"] = time.perf_counter() - t0
    res["mg_levels"] = [list(mg.level_operator(l).problem.cells) for l in range(mg.n_levels)]
    res["mg_level_dofs"] = [mg.level_operator(l).n_owned for l in range(mg.n_levels)]
    res["mg_lambda"] = {l: mg.lambda_max(l) for l in range(1, mg.n_levels)}
    solve("mg", mg)                                     # warm-up
    res["mg_cg"] = solve("mg", mg)

    # one V-cycle split by CUDA events
    h = op.initialize_dof_vector()
    mg.vmult(h, b)
    t_plain = timed(ctx, lambda: mg.vmult(h, b), reps=n_vcycles)
    mg.profile(True)
    for _ in range(n_vcycles):
        mg.vmult(h, b)
    parts, n = mg.profile_result()
    mg.profile(False)
    per = {l: {k: v / n for k, v in d.items()} for l, d in parts.items()}
    res["vcycle"] = dict(seconds_unprofiled=t_plain, ms_by_level=per,
                         ms_total_events=sum(sum(d.values()) for d in per.values()),
                         coarse_share=per[0]["coarse"] / max(1e-30, sum(sum(d.values()) for d in per.values())))

    # transfer kernels alone: algorithmic bytes (every pass reads its input once and writes its output once)
    tr = {}
    for l in range(1, mg.n_levels):
        F, Cop = mg.level_operator(l), mg.level_operator(l - 1)
        nf = [cc * p + 1 for cc in F.problem.cells]
        nc = [cc * p + 1 for cc in Cop.problem.cells]
        n_fcc, n_ffc = nf[0] * nc[1] * nc[2], nf[0] * nf[1] * nc[2]
        nbytes = 8.0 * (Cop.n_owned + 2 * n_fcc + 2 * n_ffc + F.n_owned)
        vf, vc = F.initialize_dof_vector(), Cop.initialize_dof_vector()
        mg.prolongate(l, vf, vc); mg.restrict(l, vc, vf)
        reps = max(3, int(2e9 / nbytes))
        tp = timed(ctx, lambda: mg.prolongate(l, vf, vc), reps)
        trs = timed(ctx, lambda: mg.restrict(l, vc, vf), reps)
        tr[l] = dict(bytes=nbytes, prolongate_ms=tp * 1e3, restrict_ms=trs * 1e3,
                     prolongate_GBs=nbytes / tp / 1e9, restrict_GBs=nbytes / trs / 1e9,
                     prolongate_of_copy_peak=nbytes / tp / 1e9 / COPY_PEAK_GBS,
                     restrict_of_copy_peak=nbytes / trs / 1e9 / COPY_PEAK_GBS)
        vf.close(); vc.close()
    res["transfer"] = tr
    for v in (h, b, x, diag):
        v.close()
    mg.close()
    op.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--degree", type=int, default=6)
    ap.add_argument("--cells", type=int, nargs="+", default=[88, 96])
    ap.add_argument("--tol", type=float, default=1e-8)
    ap.add_argument("--max-its", type=int, default=20000)
    ap.add_argument("--vcycles", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import dealceed_b200 as dc
    ctx = dc.Context(0)
    doc = dict(gpu_before=gpu_info(), meshes=[])
    for c in a.cells:
        doc["meshes"].append(run_mesh(dc, ctx, a.degree, c, a.tol, a.max_its, a.vcycles))
        print(json.dumps(doc["meshes"][-1]), flush=True)
    doc["gpu_after"] = gpu_info()
    ctx.close()
    text = json.dumps(doc, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
