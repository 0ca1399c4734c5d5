#!/usr/bin/env python
"""bench.py — vertices marginalised per second (SE3, fp64, NFR) on B200.

Workload (BASELINE.json configs[3], the configuration the metric is quoted on that fits one GPU):
the batched Markov-blanket sweep — synthetic SE3 blankets with n in {2,3,4,5,6,8,12,16} vertices
(H 12x12 ... 96x96 fp64), `--blankets` (default 1e5) blankets per size, star+ring edge pattern,
NFR with Chow-Liu Tree topology. One "step" = one pass of the node-removal hot path (assembly,
Schur complement, Chow-Liu MI + spanning tree, NFR closed-form information fit) over the whole
sweep. A multi-GPU run partitions the ONE sweep over the ranks (strong scaling: per size, rank r runs the r-th
contiguous slice) and gathers the substitute-edge records of every slice over NCCL/NVLink into every rank's
output buffer inside every timed step (spg_remove_round_sharded_device; the gather of one size overlaps the
kernels of the next).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--blankets B] [--impl reference] [--dump-outputs DIR]

`value`  : device-resident inputs, CUDA events on the library's stream, max over ranks; K timed steps.
`e2e`    : the same sweep through the host-buffer C-ABI call spg_remove_round (N = 1) /
           spg_remove_round_sharded (N > 1, outputs gathered to rank 0, which holds the graph):
           pinned host records in, H2D + kernels (+ gather) + D2H inside the timed region; K timed steps.
`--impl reference` times the CPU restatement of the reference path (oracle/) on all host threads
over a bounded sample of the same sweep (the reference itself cannot be built offline).
`--dump-outputs DIR` writes the output records the last device-resident timed step left in the buffers, decoded, for
a fixed seeded sample of each size's blankets (at most 64 MB): DIR/n<n>_<field>.npy, float64. The sweep is generated
from fixed seeds, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from sparsifyposegraph_b200 import records as R  # noqa: E402
from sparsifyposegraph_b200 import synth  # noqa: E402

SIZES = (2, 3, 4, 5, 6, 8, 12, 16)
VARIANT = "ring"
METRIC = "vertices marginalized/sec (SE3 fp64, NFR)"
UNIT = "vertices/s"


def workload_config(blankets, n_gpus):
    return {"workload": f"C4 batched Markov-blanket sweep: SE3, n in {list(SIZES)}, {blankets} blankets per size per GPU, "
                        f"star+ring edges, NFR Chow-Liu tree (closed-form fit)",
            "blankets_per_size": blankets, "sizes": list(SIZES), "topology": "tree", "algorithm": "nfr",
            "lin_point": "global", "l2": "inputs larger than L2 (126 MB) at the default size; each blanket is read once",
            "parallelism": (f"one sweep partitioned over {n_gpus} GPU(s) (strong scaling); per step every rank's substitute-edge "
                            f"records are gathered over NCCL/NVLink into every rank's output buffer, inside the timed region"
                            if n_gpus > 1 else "1 GPU")}


def make_sweep(blankets, rank):
    sweep = []
    for n in SIZES:
        blk = synth.make_blankets(n, blankets, dim=6, variant=VARIANT, seed=synth.SEED + n)  # the same sweep on every rank
        nk = np.full(blankets, n - 1, dtype=np.int64)
        blk["out_off"] = R.out_offsets(6, R.ALG_NFR, R.TOPO_TREE, 1.0, nk)
        sweep.append(blk)
    return sweep


DUMP_BYTES = 60 << 20   # --dump-outputs: the arrays of all sizes together (the .npy headers stay within 64 MB)
DUMP_SEED = 20261020


def sample_outputs(dev, sweep):
    """The device output buffers of every size, decoded for the same seeded sample of blankets in every run: blanket index,
    status, number of new edges, KLD, and per substitute edge its vertex pair, measurement and information matrix."""
    import torch
    n_edges = {d["n"]: R.out_edge_count(R.ALG_NFR, R.TOPO_TREE, 1.0, d["n"] - 1) for d in dev}
    per_blanket = 8 * sum(4 + ne * (2 + R.pose_words(6) + 36) for ne in n_edges.values())
    k = DUMP_BYTES // per_blanket
    rng = np.random.default_rng(DUMP_SEED)
    arrays = {}
    for d, blk in zip(dev, sweep):
        n, B, ne = d["n"], d["B"], n_edges[d["n"]]
        idx = np.arange(B) if k >= B else np.sort(rng.choice(B, k, replace=False))
        W = int(blk["out_off"][1] - blk["out_off"][0])   # uniform blankets: one record size per size
        words = torch.from_numpy(blk["out_off"][idx][:, None] + np.arange(W)).cuda()
        rec = d["out"][words].cpu().numpy().view(np.uint64)
        status, pairs, meas, info = R.nfr_uniform_view(rec.reshape(-1), np.arange(len(idx) + 1) * W, 6, n - 1, ne)
        arrays.update({f"n{n}_blanket": idx, f"n{n}_status": status, f"n{n}_n_new_edges": rec.view(np.int32)[:, 1],
                       f"n{n}_kld": rec.view(np.float64)[:, 2]})
        if ne:
            arrays.update({f"n{n}_pairs": pairs, f"n{n}_meas": meas, f"n{n}_info": info})
    return {name: np.ascontiguousarray(a, dtype=np.float64) for name, a in arrays.items()}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.samples.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
            except Exception:
                continue
            for nme, v in zip(names, s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args, rank, world):
    """CPU arm: the oracle (restatement of the reference's CPU path) on all host threads."""
    if rank != 0:
        return
    from oracle import pyoracle
    pyoracle.build()
    cores = os.cpu_count() or 1
    S = args.ref_sample
    sweep = []
    for n in SIZES:
        blk = synth.make_blankets(n, S, dim=6, variant=VARIANT, seed=synth.SEED + n)
        blk["out_off"] = R.out_offsets(6, R.ALG_NFR, R.TOPO_TREE, 1.0, np.full(S, n - 1))
        sweep.append(blk)
    opts = pyoracle.make_opts(R.TOPO_TREE, R.LIN_GLOBAL, 1.0)

    def step():
        t = 0.0
        for blk in sweep:
            _, secs, _, _ = pyoracle.remove_round(6, R.ALG_NFR, opts, blk["records"], blk["rec_off"], blk["out_off"], cores)
            t += secs
        return t
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    total = len(SIZES) * S * args.steps
    val = total / dt
    sample = f"first {S} blankets of each of the {len(SIZES)} sizes per step (same generator and mix as the GPU arm)"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args.blankets, args.gpus),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "note": "CPU restatement of the reference path (oracle/); the reference itself needs "
                                     "Eigen/g2o/iSAM/CHOLMOD and cannot be built offline"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


_JSON_OUT = None


def _claim_stdout():
    """The driver reads ONE JSON line from stdout. Libraries write there too (NCCL prints its version banner at
    NCCL_DEBUG >= VERSION): keep a private copy of fd 1 for the JSON line and point fd 1 at stderr for everyone else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    _claim_stdout()
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--blankets", type=int, default=100000, help="blankets per size per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-sample", type=int, default=256, help="blankets per size per step for the CPU arms")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sizes", default=None, help="comma list overriding the size sweep (debug)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed, seeded sample of the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    global SIZES
    if args.sizes:
        SIZES = tuple(int(x) for x in args.sizes.split(","))

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from sparsifyposegraph_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the node-removal path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    os.environ["NCCL_DEBUG"] = os.environ.get("SPG_NCCL_DEBUG", "INFO" if world > 1 else "WARN")  # INFO: the driver counts ranks
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = capi.Context(local_rank)
    if world > 1:
        from sparsifyposegraph_b200 import distributed
        distributed.init_comm(ctx, rank, world)  # the library's own NCCL communicator (spg_comm_init)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))
    opts = capi.make_opts(R.TOPO_TREE, R.LIN_GLOBAL, 1.0, flags=2)  # SPG_OPT_POSE_EDGES_ONLY: the sweep has POSE edges only

    # ---- data: per-size device-resident records + one mixed host round for the e2e path -------------
    sweep = make_sweep(args.blankets, rank)
    dev = []
    for blk in sweep:
        d = {"n": blk["n"], "E": blk["E"], "B": blk["B"],
             "rec": torch.from_numpy(blk["records"].view(np.int64)).cuda(),
             "rec_off": torch.from_numpy(blk["rec_off"]).cuda(),
             "out_off": torch.from_numpy(blk["out_off"]).cuda(),
             "out": torch.zeros(int(blk["out_off"][-1]), dtype=torch.int64, device="cuda")}
        dev.append(d)
    total_blankets = sum(b["B"] for b in sweep)
    # mixed host round (all sizes in one spg_remove_round call), pinned
    rec_words = sum(len(b["records"]) for b in sweep)
    out_words = sum(int(b["out_off"][-1]) for b in sweep)
    h_rec = torch.empty(rec_words, dtype=torch.int64).pin_memory()
    h_out = torch.empty(out_words, dtype=torch.int64).pin_memory()
    h_rec_np = h_rec.numpy().view(np.uint64)
    h_out_np = h_out.numpy().view(np.uint64)
    rec_off_all = np.zeros(total_blankets + 1, dtype=np.int64)
    out_off_all = np.zeros(total_blankets + 1, dtype=np.int64)
    pr = po = pb = 0
    for b in sweep:
        n_r, n_o, nb = len(b["records"]), int(b["out_off"][-1]), b["B"]
        h_rec_np[pr:pr + n_r] = b["records"]
        rec_off_all[pb:pb + nb + 1] = b["rec_off"] + pr
        out_off_all[pb:pb + nb + 1] = b["out_off"] + po
        pr += n_r
        po += n_o
        pb += nb
    h2d_bytes = rec_words * 8 + 2 * (total_blankets + 1) * 8 + total_blankets * 4
    d2h_bytes = out_words * 8

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # per size: rank r runs blankets [B r / N, B (r+1) / N) and every rank receives all slices (uniform blankets: equal
    # counts are cost-balanced). Largest blankets first, so the gather left exposed at the end of a step is the smallest.
    for d, blk in zip(dev, sweep):
        d["bounds"] = np.array([d["B"] * r // world for r in range(world + 1)], dtype=np.int32)
        d["wbounds"] = blk["out_off"][d["bounds"]].astype(np.int64)
    order = sorted(dev, key=lambda d: -d["n"])

    def device_step():
        for d in order:
            if world == 1:
                ctx.remove_round_device(6, R.ALG_NFR, opts, d["B"], d["rec"].data_ptr(), d["rec_off"].data_ptr(),
                                        d["out_off"].data_ptr(), d["out"].data_ptr(), d["n"], d["E"])
            else:
                ctx.remove_round_sharded_device(6, R.ALG_NFR, opts, d["B"], d["rec"].data_ptr(), d["rec_off"].data_ptr(),
                                                d["out_off"].data_ptr(), d["out"].data_ptr(), d["bounds"], d["wbounds"],
                                                d["n"], d["E"], root=-1)
        if world > 1:
            ctx.comm_join()  # the compute stream waits for the step's gathers: the output buffers are complete (and reusable)

    # ---- FP64 peak (roofline denominator; MEASURED_PEAKS.json has no FP64 figure) --------------------
    fp64_peak = ctx.fp64_peak_tflops(5)

    # ---- warm-up ------------------------------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        device_step()
    ctx.sync()
    barrier()

    # ---- timed: device-resident ---------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(stream):
        ev0.record()
        for _ in range(args.steps):
            device_step()
        ev1.record()
    ctx.sync()  # compute stream and the gather stream
    barrier()
    dev_ms = ev0.elapsed_time(ev1)  # every step ends with comm_join: ev1 is behind the last gather too
    launches = ctx.launches - launches0
    dumped = sample_outputs(dev, sweep) if args.dump_outputs and rank == 0 else None  # before the per-size pass below
    # every blanket of the whole sweep must be present and OK in THIS rank's output buffers (own slice from the
    # kernels, the other slices through the gather): status == 0 and n_new_edges == n - 2
    n_dev_ok = 0
    for d, blk in zip(dev, sweep):
        hdr = d["out"][torch.from_numpy(blk["out_off"][:-1]).cuda()].cpu().numpy().view(np.int32).reshape(-1, 2)
        n_dev_ok += int(((hdr[:, 0] == 0) & (hdr[:, 1] == d["n"] - 2)).sum())

    # per-size kernel time (dominant kernel + roofline), one extra pass, events on the same stream
    per_size = []
    for d in dev:
        nb_mine = int(d["bounds"][rank + 1] - d["bounds"][rank])
        b0 = int(d["bounds"][rank])
        with torch.cuda.stream(stream):
            a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ctx.remove_round_device(6, R.ALG_NFR, opts, nb_mine, d["rec"].data_ptr(), d["rec_off"].data_ptr() + 8 * b0,
                                    d["out_off"].data_ptr() + 8 * b0, d["out"].data_ptr(), d["n"], d["E"])
            b2.record()
        ctx.sync()
        ms = a.elapsed_time(b2)
        alg = synth.algorithmic_bytes_flops(d["n"], d["E"], 6, "nfr")
        per_size.append({"n": d["n"], "E": d["E"], "ms": ms, "blankets": nb_mine, "vertices_per_s": nb_mine / (ms * 1e-3),
                         "gflops": alg["flops"] * nb_mine / (ms * 1e-3) / 1e9,
                         "gbs": alg["bytes"] * nb_mine / (ms * 1e-3) / 1e9})
    clocks = sampler.stop()

    # ---- timed: end to end through the host-buffer C ABI ----------------------------------------------
    e2e_steps = args.steps   # the same K as the device-resident loop (~0.13 s per step)
    shard_info = None
    e2e_modes = {}
    shm = None
    if world > 1:
        # host-resident graph on one node: ONE output buffer in POSIX shared memory, mapped and page-locked by every rank;
        # each rank copies the records of its own blankets into it over its own PCIe link (SPG_ROOT_SHARED_HOST)
        from multiprocessing import shared_memory
        name = [f"spg_bench_out_{os.getpid()}" if rank == 0 else None]
        if rank == 0:
            shm = shared_memory.SharedMemory(name=name[0], create=True, size=out_words * 8)
        dist.broadcast_object_list(name, src=0)
        if rank != 0:
            shm = shared_memory.SharedMemory(name=name[0])
        sh_out_np = np.ndarray((out_words,), dtype=np.uint64, buffer=shm.buf)
        rc = torch.cuda.cudart().cudaHostRegister(sh_out_np.ctypes.data, out_words * 8, 0)
        assert int(rc) == 0, f"cudaHostRegister failed: {rc}"

    def e2e_call(mode):
        nonlocal shard_info
        if world == 1:
            ctx.remove_round(6, R.ALG_NFR, opts, h_rec_np, rec_off_all, out_off_all, out=h_out_np)
        elif mode == "shared_host":   # collective; every rank writes its slices of the one host buffer, then the ranks meet
            _, shard_info = ctx.remove_round_sharded(6, R.ALG_NFR, opts, h_rec_np, rec_off_all, out_off_all, out=sh_out_np, root=-2)
            dist.barrier()
        else:                         # NCCL gather of the records to rank 0 over NVLink, rank 0 copies everything to its host buffer
            _, shard_info = ctx.remove_round_sharded(6, R.ALG_NFR, opts, h_rec_np, rec_off_all, out_off_all, out=h_out_np, root=0)

    def count_ok(buf):
        hdr = buf[out_off_all[:-1]].view(np.int32).reshape(-1, 2)
        nk_all = np.concatenate([np.full(b["B"], b["n"] - 2) for b in sweep])
        return int(((hdr[:, 0] == 0) & (hdr[:, 1] == nk_all)).sum())

    n_ok = 0
    for mode in (["host"] if world == 1 else ["nccl_root0", "shared_host"]):
        buf = h_out_np if mode != "shared_host" else sh_out_np
        if rank == 0:
            buf[:] = 0
        barrier()
        e2e_call(mode)  # warm-up (allocations)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_call(mode)
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        barrier()
        ok = count_ok(buf) if rank == 0 else 0
        e2e_modes[mode] = {"seconds": secs, "blankets_ok": ok,
                           "h2d": shard_info["h2d_bytes"] if shard_info else h2d_bytes,
                           "d2h": shard_info["d2h_bytes"] if shard_info else d2h_bytes,
                           "gather_window_ms": shard_info["gather_window_ms"] if shard_info else None}
    headline = "host" if world == 1 else "shared_host"
    e2e_s, n_ok = e2e_modes[headline]["seconds"], e2e_modes[headline]["blankets_ok"]
    h2d_bytes, d2h_bytes = e2e_modes[headline]["h2d"], e2e_modes[headline]["d2h"]
    # ---- reduce over ranks ----------------------------------------------------------------------------
    gather = None
    if world > 1:
        t = torch.tensor([dev_ms, e2e_s, e2e_modes["nccl_root0"]["seconds"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_s, nccl_s = float(t[0]), float(t[1]), float(t[2])
        t = torch.tensor([n_dev_ok, h2d_bytes, d2h_bytes, e2e_modes["nccl_root0"]["h2d"], e2e_modes["nccl_root0"]["d2h"]], dtype=torch.int64, device="cuda")
        tmin = t.clone()
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        n_dev_ok = int(tmin[0])          # the worst rank's count of complete, OK blankets in its gathered buffers
        h2d_bytes, d2h_bytes = int(t[1]), int(t[2])  # whole job
        gather = {"all_gather_bytes_per_step_per_rank": int(sum(int(b["out_off"][-1]) for b in sweep) * 8 * (world - 1) // world),
                  "e2e_mode": "SPG_ROOT_SHARED_HOST: every rank copies its own records into one shared, page-locked host buffer",
                  "e2e_nccl_gather_to_rank0": {"value": total_blankets * e2e_steps / nccl_s, "unit": UNIT,
                                               "blankets_ok": e2e_modes["nccl_root0"]["blankets_ok"],
                                               "h2d_bytes_per_step": int(t[3]), "d2h_bytes_per_step": int(t[4]),
                                               "gather_window_ms_rank0": e2e_modes["nccl_root0"]["gather_window_ms"],
                                               "note": "rank 0 reads ALL records back over its own PCIe link: bound by that copy"},
                  "e2e_pipeline_steps": shard_info["steps"] if shard_info else None}
    if shm is not None:
        torch.cuda.cudart().cudaHostUnregister(sh_out_np.ctypes.data)
        del sh_out_np
        shm.close()
        if rank == 0:
            shm.unlink()
    if rank == 0:
        value = total_blankets * args.steps / (dev_ms * 1e-3)   # the one sweep, whatever the number of ranks
        e2e_value = total_blankets * e2e_steps / e2e_s
        dom = max(per_size, key=lambda p: p["ms"])
        alg = synth.algorithmic_bytes_flops(dom["n"], dom["E"], 6, "nfr")
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        tiles = (dom["n"] - 1) * dom["n"] // 2   # launch_dim<6> in csrc/spg_capi.cu picks the instantiation by the blanket's tile count
        kname = ("blanket_kernel<6,32>" if dom["n"] < 3 else "fast_kernel<6,8,1>" if tiles <= 8 else "fast_kernel<6,16,1>" if tiles <= 16 else
                 "fast_kernel<6,32,1>" if tiles <= 32 else "fast_kernel<6,0,4>" if tiles <= 128 else "fast_kernel<6,0,8>")
        roofline = {"bound": "fp64", "kernel": f"{kname} (n={dom['n']} bucket)",
                    "achieved": dom["gflops"] / 1e3, "peak": fp64_peak, "unit": "TFLOP/s",
                    "frac": dom["gflops"] / 1e3 / fp64_peak if fp64_peak else None,
                    "peak_source": "measured here: register-resident DFMA loop on all SMs (spg_fp64_peak_probe); "
                                   "MEASURED_PEAKS.json has no FP64 figure",
                    "algorithmic_flops_per_blanket": alg["flops"], "algorithmic_bytes_per_blanket": alg["bytes"],
                    "hbm": {"achieved": dom["gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": dom["gbs"] / hbm_peak,
                            "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback"},
                    "traffic": None, "share_of_step": dom["ms"] / sum(p["ms"] for p in per_size)}
        try:  # DRAM bytes per blanket of this kernel from the committed ncu --set full capture
            tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            if tr.get("n") == dom["n"]:
                roofline["traffic"] = tr["dram_bytes_per_blanket"] * dom["blankets"]
                roofline["traffic_source"] = tr["source"]
                # the contract's `frac` counts the reference algorithm's flops; what the FP64 pipe really executed:
                roofline["fp64_pipe_active_pct_ncu"] = tr.get("fp64_pipe_active_pct")
                roofline["fp64_pipe_source"] = tr.get("fp64_pipe_source")
        except Exception:
            pass
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": workload_config(args.blankets, world),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                        "steps": e2e_steps, "blankets_ok": n_ok, "blankets": total_blankets},
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "per_size": per_size,
                "fp64_peak_tflops_measured": fp64_peak, "gather": gather,
                "blankets_ok_device": n_dev_ok, "blankets_total": total_blankets}
        assert n_dev_ok == total_blankets, f"device-resident outputs: only {n_dev_ok} of {total_blankets} blankets complete and OK"
        if not args.no_cpu_baseline:
            from oracle import pyoracle
            pyoracle.build()
            cores = os.cpu_count() or 1
            S = args.ref_sample
            o_opts = pyoracle.make_opts(R.TOPO_TREE, R.LIN_GLOBAL, 1.0)
            secs = 0.0
            for blk in sweep:
                W = int(blk["rec_off"][1])
                nb = min(S, blk["B"])
                _, s, _, _ = pyoracle.remove_round(6, R.ALG_NFR, o_opts, blk["records"][: nb * W], blk["rec_off"][: nb + 1],
                                                   blk["out_off"][: nb + 1], cores)
                secs += s
            nb_total = sum(min(S, blk["B"]) for blk in sweep)
            line["cpu_baseline"] = {"value": nb_total / secs, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"first {S} blankets of each size of this run's sweep, one blanket per thread"}
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
            line["dump_outputs"] = {"dir": args.dump_outputs, "arrays": len(dumped),
                                    "bytes": sum(a.nbytes for a in dumped.values()),
                                    "blankets_per_size": len(dumped[f"n{SIZES[0]}_blanket"])}
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
