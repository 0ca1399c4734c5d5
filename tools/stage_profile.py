#!/usr/bin/env python
"""Per-stage cycle breakdown of the blanket kernels (clock64 accumulators, thread 0 of every CTA).
usage: stage_profile.py [n ...]   (SE3, NFR tree, ring blankets). SPG_NO_FAST=1 profiles blanket_kernel;
SPG_PROF_ALG=1 profiles the GLC tree path."""
import ctypes as C
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sparsifyposegraph_b200 import capi, records as R, synth  # noqa: E402

NAMES = ["load", "assembly", "schur", "cl_chol", "cl_inverse", "cl_blockchol", "cl_mi", "kruskal", "g_chol", "g_inverse",
         "new_jac", "sigma", "x_inv", "glc get_edge+write", "glc marginal", "glc pinv+target"]
FAST = ["load+poses", "asm: H_k0, H_00", "schur", "C (+G) sweep", "MI weights", "kruskal", "G sweep / guards", "closed form",
        "asm: Jacobians", "asm: Omega J", "asm: wait for the other edges", "asm: block gather"] + ["-"] * 4
sizes = [int(x) for x in sys.argv[1:]] or [5, 16]
ctx = capi.Context(0)
L = capi.lib()
L.spg_stage_profile.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
for n in sizes:
    B = int(os.environ.get("SPG_PROF_B", "8000")) if n <= 19 else 8
    blk = synth.make_blankets(n, B, dim=6, variant="ring", seed=n)
    ALG = int(os.environ.get("SPG_PROF_ALG", "0"))
    out_off = R.out_offsets(6, ALG, 0, 1.0, np.full(B, n - 1))
    ctx.remove_round(6, ALG, capi.make_opts(0, 1), blk["records"], blk["rec_off"], out_off)
    L.spg_stage_profile(ctx.h, 1, None)
    ctx.remove_round(6, ALG, capi.make_opts(0, 1), blk["records"], blk["rec_off"], out_off)
    retried = ctx.last_retry_count
    cyc = np.zeros(32, dtype=np.uint64)
    L.spg_stage_profile(ctx.h, 0, cyc.ctypes.data_as(C.c_void_p))
    print(f"n={n}: kernel {ctx.last_kernel_ms:.3f} ms for {B} blankets, {retried} handed to blanket_kernel")
    for label, names, c16 in (("blanket_kernel", NAMES, cyc[:16]), ("fast_kernel", FAST, cyc[16:])):
        tot = c16.sum()
        if not tot:
            continue
        print(f"  {label}: {tot / B:.0f} cycles per blanket (thread 0 view)")
        for nm, c in zip(names, c16):
            if c:
                print(f"   {nm:14s} {c / B:10.0f} cyc  {100.0 * c / tot:5.1f}%")
