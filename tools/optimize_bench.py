"""spg_graph_optimize on graphs beyond the dense path's limit (block-sparse BSR + block-Jacobi PCG), one GPU.

    python tools/optimize_bench.py [--rows 1000 --cols 1000] [--mid 300] [--max-iterations 10] [--out FILE]

Graphs (synthetic SE3 grids of synth.make_grid_graph, noisy measurements, estimates at the generating poses, vertex 0
fixed as in GraphWrapperG2O::optimize):
  grid RxC before removal        BASELINE.json configs[4] as generated (1 M poses: 6 M dimensions);
  grid RxC after removal         the same grid after globalDecimate's removal at sparsity 10 (NFR Tree), the graph the
                                 reference's marginalize() optimises next;
  grid MxM                       a mid-size grid (default 300 x 300);
  sphere dense / sparse          A/B of the two solvers on sphere.g2o, the sparse one forced by SPG_OPT_DENSE_MAX_DIMS
                                 (information only: the dense path runs wherever it fits).
Each graph: wall time of the optimize call (host clock; the call ends synchronised), LM iterations and trials, PCG
iterations, then a second, profiled call of one LM iteration (torch.profiler, CUDA activities) for the device time of
the PCG kernels per CG iteration and the BSR bytes (block values + column indices + row pointers) the SpMV streams per
iteration over the SpMV's time, against the 7.7 TB/s HBM3e data-sheet figure. max_iterations defaults to 10 (the
reference uses 50) to bound the run; the per-iteration figures do not depend on it.
Prints one JSON line per graph and writes them all, with the card's name and power limit read in the same run, to
--out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from sparsifyposegraph_b200 import capi, records as R, synth  # noqa: E402

HBM_DATASHEET_TBS = 7.7
PCG_KERNELS = ("pcg_spmv_dot_kernel", "pcg_alpha_kernel", "pcg_update_kernel", "pcg_beta_kernel")


def bsr_bytes(dim, n_free_vertices, pairs):
    """Bytes of the BSR arrays the SpMV reads once per CG iteration. pairs: (E, 2) distinct-vertex factor pairs of free
    vertices (pose edges); both triangles are stored, plus every diagonal block."""
    p = np.sort(np.asarray(pairs, dtype=np.int64), axis=1)
    nnzb = n_free_vertices + 2 * len(np.unique(p[:, 0] * (1 << 32) + p[:, 1]))
    return nnzb * (dim * dim * 8 + 4) + (n_free_vertices + 1) * 4, nnzb


def profile_pcg(ctx, g, fixed):
    """One LM iteration under torch.profiler: device time of each PCG kernel (ms) and the CG iterations it ran."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        st = g.optimize(ctx, fixed=fixed, max_iterations=1)
        torch.cuda.synchronize()
    ms = {}
    for ev in prof.key_averages():
        for k in PCG_KERNELS:
            if k in ev.key:
                t = getattr(ev, "device_time_total", None)
                if t is None:
                    t = ev.cuda_time_total
                ms[k] = ms.get(k, 0.0) + t / 1e3
    return ms, st["cg_iterations"]


def run(ctx, label, g, fixed, max_iterations, pairs, hook=None):
    if hook is None:
        os.environ.pop("SPG_OPT_DENSE_MAX_DIMS", None)
    else:
        os.environ["SPG_OPT_DENSE_MAX_DIMS"] = str(hook)
    t0 = time.time()
    st = g.optimize(ctx, fixed=fixed, max_iterations=max_iterations)
    wall = time.time() - t0
    rec = {"graph": label, "wall_s": wall, "dimensions": st["dimensions"], "solver": "sparse_pcg" if st["solver"] else "dense_cholesky",
           "lm_iterations": st["iterations"], "lm_trials": st["trials"], "cg_iterations": st["cg_iterations"],
           "cg_max_rel_residual": st["cg_max_rel_residual"], "chi2_initial": st["chi2_initial"], "chi2_final": st["chi2_final"],
           "max_iterations": max_iterations}
    if st["solver"] == 1:
        nb = st["dimensions"] // g.dim
        nbytes, nnzb = bsr_bytes(g.dim, nb, pairs)
        ms, iters = profile_pcg(ctx, g, fixed)
        rec.update({"bsr_blocks": nnzb, "bsr_bytes": nbytes, "profiled_cg_iterations": iters,
                    "device_ms_per_cg_iteration": sum(ms.values()) / max(iters, 1),
                    "spmv_ms_per_cg_iteration": ms.get("pcg_spmv_dot_kernel", 0.0) / max(iters, 1),
                    "pcg_kernel_ms": ms})
        spmv_s = rec["spmv_ms_per_cg_iteration"] * 1e-3
        it_s = rec["device_ms_per_cg_iteration"] * 1e-3
        rec["spmv_bsr_TBs"] = nbytes / spmv_s / 1e12 if spmv_s > 0 else None
        rec["iteration_bsr_TBs"] = nbytes / it_s / 1e12 if it_s > 0 else None
        rec["hbm_datasheet_TBs"] = HBM_DATASHEET_TBS
    os.environ.pop("SPG_OPT_DENSE_MAX_DIMS", None)
    print(json.dumps(rec), flush=True)
    return rec


def free_pairs(g, fixed):
    fx = set(fixed)
    pairs = [(int(e["v"][0]), int(e["v"][1])) for e in g.edges() if e["kind"] == 0]
    return [p for p in pairs if p[0] not in fx and p[1] not in fx]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1000)
    ap.add_argument("--cols", type=int, default=1000)
    ap.add_argument("--mid", type=int, default=300)
    ap.add_argument("--sparsity", type=int, default=10)
    ap.add_argument("--max-iterations", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("optimize_bench.py needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card:", card, flush=True)
    ctx = capi.Context(0)
    fixed = (0,)
    # warm-up: module load, first launches of both paths
    w = synth.fill_graph(capi.Graph(dim=6), *synth.make_grid_graph(10, 10, dim=6))
    w.optimize(ctx, max_iterations=2)
    os.environ["SPG_OPT_DENSE_MAX_DIMS"] = "0"
    w.optimize(ctx, max_iterations=2)
    os.environ.pop("SPG_OPT_DENSE_MAX_DIMS")
    recs = []

    def grid(rows, cols):
        data = synth.make_grid_graph(rows, cols, dim=6)
        e = data[1]
        return synth.fill_graph(capi.Graph(dim=6), *data), e[(e[:, 0] != 0) & (e[:, 1] != 0)]

    g, pairs = grid(args.mid, args.mid)
    recs.append(run(ctx, f"grid {args.mid}x{args.mid}", g, fixed, args.max_iterations, pairs))
    del g
    g, pairs = grid(args.rows, args.cols)
    recs.append(run(ctx, f"grid {args.rows}x{args.cols} before removal", g, fixed, args.max_iterations, pairs))
    del g
    g, _ = grid(args.rows, args.cols)
    which = synth.grid_removal_order(args.rows, args.cols, args.sparsity, 4, "random")
    g.marginalize(ctx, which, capi.make_opts(R.TOPO_TREE, R.LIN_GLOBAL), R.ALG_NFR)
    recs.append(run(ctx, f"grid {args.rows}x{args.cols} after removal (sparsity {args.sparsity}, NFR Tree)", g, fixed,
                    args.max_iterations, free_pairs(g, fixed)))
    del g
    import datasets
    for hook in (None, 0):
        g = capi.Graph(datasets.path("sphere"))
        recs.append(run(ctx, "sphere " + ("dense" if hook is None else "sparse (forced)"), g, fixed, 50, free_pairs(g, fixed), hook))
    ctx.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps({"card": card, "power_limit_and_max_sm_clock_from": "nvidia-smi in the same run"}) + "\n")
            for r in recs:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
