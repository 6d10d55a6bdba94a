"""Device time per kernel of one merged-CG iteration, from torch.profiler (CUPTI) over whole solves.

    python scripts/cg_kernel_times.py --label new --out profiles/x.json [--degree 6 --cells 88 --its 40]
    BP5_LIB=<other libbp5b200.so> python scripts/cg_kernel_times.py --label old ...   # another build, same ABI

The solve runs with per-launch events on (bp5_operator_profile), so the CUDA graph is off and every kernel is its own
activity; kernels are grouped by name (template arguments dropped) and their summed device time is divided by the
iterations.  Run it in a process of its own: the profiler slows the host, so these are not headline numbers."""
import argparse
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def short(name):
    name = re.sub(r"^void ", "", name)
    name = re.sub(r"<.*", "", name)
    return name.replace("bp5::", "")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--degree", type=int, default=6)
    ap.add_argument("--cells", type=int, default=88)
    ap.add_argument("--quadrature", choices=("gll", "gauss"), default="gll")
    ap.add_argument("--its", type=int, default=40)
    ap.add_argument("--label", default="")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import dealceed_b200 as dc

    ctx = dc.Context(0)
    quad = dc.QUAD_GLL if a.quadrature == "gll" else dc.QUAD_GAUSS
    op = dc.PoissonOperator(ctx, dc.make_problem(a.degree, (a.cells,) * 3, quadrature=quad, deformation=0))
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    op.do_zero_out = False
    control = dc.IterationNumberControl(a.its, 1e-6 * b.l2_norm())
    solver = dc.SolverCGFullMerge(control)
    op.profile(True)
    x.set(0.0)
    solver.solve(op, x, b, history=False)            # warm-up: module loads, kernel attributes
    ctx.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        x.set(0.0)
        solver.solve(op, x, b, history=False)
        ctx.synchronize()
    its = control.last_step()
    op.profile(False)
    per = {}
    for e in prof.events():
        if e.device_type.name != "CUDA" or not e.name or e.name.startswith("Memcpy"):
            continue
        k = short(e.name)
        t = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
        d = per.setdefault(k, {"calls": 0, "us": 0.0})
        d["calls"] += 1
        d["us"] += t
    rows = {k: {"calls_per_it": v["calls"] / its, "ms_per_it": v["us"] / its / 1e3} for k, v in per.items()}
    out = {"label": a.label, "lib": os.environ.get("BP5_LIB", "this tree"), "gpu": torch.cuda.get_device_name(0),
           "workload": f"BP5 p={a.degree} {a.quadrature}, {a.cells}^3 cells, undeformed (stored metric), merged CG, {its} iterations",
           "n_dofs": op.n_owned, "iterations": its, "kernels": rows,
           "total_ms_per_it": sum(r["ms_per_it"] for r in rows.values()),
           "note": "per-solve kernels (permutations, initial residual, finish) are spread over the iterations"}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    for k, r in sorted(rows.items(), key=lambda kv: -kv[1]["ms_per_it"]):
        print(f"{a.label:5s} {k:40s} {r['calls_per_it']:6.2f} calls/it {r['ms_per_it']:8.4f} ms/it")
    print(f"{a.label:5s} total {out['total_ms_per_it']:.4f} ms/it")
    b.close(); x.close(); op.close(); ctx.close()


if __name__ == "__main__":
    main()
