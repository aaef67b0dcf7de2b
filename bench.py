#!/usr/bin/env python
"""Benchmark of the rigid-ICP hot path (BASELINE.json metric: ICP iterations/s and correspondences/s).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--no-secondary]
                    [--dump-outputs DIR]

A "step" is one full ICP iteration (transform + radius-bounded 1-NN of every source point + moment accumulation +
reduction (+ all-reduce) + solve) on the named workload.

  N = 1  BASELINE.json configs[1]: 1 M -> 1 M synthetic uniform clouds, point-to-point metric, k = 1 (`icp_p2p_1m`).
         The same JSON line carries a `secondary` block with the other single-GPU configs (configs[2] on one GPU:
         10 M -> 10 M combined metric; configs[3]: KMeans3f 50 M x 1024; configs[4]: RANSAC scoring 5 M pairs; PCA 50 M).
  N > 1  BASELINE.json configs[2], STRONG-scaled (one process per GPU under torchrun): 10 M destination points +
         normals replicated on every rank, the 10 M source points split into N contiguous shards, combined metric
         (w_pt 0.1, w_pl 1), max_distance^2 = 0.01^2. The only exchange per iteration is the all-reduce of the 28
         normal-equation values, done over NVLink peer memory by the iteration's one-warp finish kernel. `secondary`
         carries KMeans3f 50 M x 1024 sharded over the N ranks. (The N = 1 point of this strong-scaling curve is
         `secondary.icp_combined_10m` of the N = 1 line.)

`value` counts correspondences (source points processed) per second over ALL ranks; iterations/s is next to it.

Timing: W untimed warm-up iterations (a separate estimate() call), then ONE estimate() call of exactly K iterations
(tol = 0) bracketed by barrier + synchronize; every iteration is timed on the device with a CUDA-event pair around
the iteration's kernels, with an L2 flush (256 MiB memset) before every iteration OUTSIDE the event bracket; max over
ranks. The timed call starts like every ICP run: its first iteration searches every query (nothing cached), later
iterations re-search only the queries whose cached match cannot be proven to still be the nearest neighbour
(icp_loop.cu) - `roofline` reports the mean and both regimes.
--dump-outputs DIR writes what that timed call returned after its last step (DIR/T.npy, the 3 x 4 float32 transform,
and the float64 scalars DIR/num_corr.npy, iterations.npy, last_delta.npy, converged.npy); the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
Parity inside the bench: the GPU transform is compared with the CPU arm's (same inputs, same iteration count), the
correspondence counts must be equal, all ranks must hold bit-identical transforms, and at N > 1 the sharded result
is compared with a single-GPU run of the whole problem on rank 0.
The reference arm (--impl reference) times cilantro's own CPU path: the reference's vendored nanoflann compiled in
place (oracle/_ref) driving the Eigen-free restatement of its ICP loop (oracle/), on all host cores. Nothing here
reads /root/reference at run time.
"""
import argparse
import hashlib
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

WORKLOADS = {
    # name: points, metric, with normals, max_d2, icp kwargs, iterations of one estimate() call (SURVEY 8d)
    "icp_p2p_1m": dict(n=1_000_000, metric="p2p", normals=False, max_d2=0.02 ** 2, kw={}, iters=15),
    "icp_combined_10m": dict(n=10_000_000, metric="combined", normals=True, max_d2=0.01 ** 2,
                             kw=dict(w_pt=0.1, w_pl=1.0), iters=10),
    "icp_p2p_100k": dict(n=100_000, metric="p2p", normals=False, max_d2=0.05 ** 2, kw={}, iters=15),
    "icp_combined_200k": dict(n=200_000, metric="combined", normals=True, max_d2=0.04 ** 2,
                              kw=dict(w_pt=0.1, w_pl=1.0), iters=10),
}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(workload):
    """dram bytes per ICP iteration (cold / warm) from the committed ncu --set full captures."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get(workload)
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(smax)) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_inputs(w, rank, world, scaling, pinned=False, survey_pose=False):
    """Seeded synthetic pair. weak: dst = world * n points (replicated), every rank's src shard = n points.
    strong: dst = n points (replicated), src = n points split into `world` contiguous shards.
    survey_pose: SURVEY 8(d)'s fixed generating pose (0.02 rad) instead of the spacing-scaled one (synth.t_ref_for)."""
    from cilantro_b200 import synth
    from cilantro_b200.dist import shard_bounds

    n_total = w["n"] * world if scaling == "weak" else w["n"]
    dst, src, nrm, T_ref = synth.icp_pair(n_total, seed=1, noise=0.001, with_normals=w["normals"],
                                          T_ref=synth.t_ref_default() if survey_pose else None)
    lo, hi = shard_bounds(n_total, rank, world)
    src_all = src
    src = np.ascontiguousarray(src[lo:hi])
    keep = None
    if pinned:
        import torch

        def pin(a):
            if a is None:
                return None
            t = torch.empty(a.shape, dtype=torch.float32, pin_memory=True)
            t.numpy()[...] = a
            return t

        keep = [pin(dst), pin(src), pin(nrm)]
        dst, src, nrm = keep[0].numpy(), keep[1].numpy(), (keep[2].numpy() if keep[2] is not None else None)
    return dict(dst=dst, src=src, nrm=nrm, T_ref=T_ref, lo=lo, keep=keep, src_all=src_all, n_total=n_total)


def cpu_reference_run(w, steps, warmup, dst, src, nrm, build_in_timed_region):
    """cilantro's CPU path on the host cores: reference nanoflann (oracle/_ref) + restated ICP loop."""
    import oracle

    oracle.build()
    kind = "reference" if oracle.have_ref() else "port"
    mk = (lambda: oracle.RefKnn(dst)) if oracle.have_ref() else (lambda: oracle.BruteKnn(dst))
    kw = dict(metric=w["metric"], dst_n=nrm, tol=0.0, max_d2=np.float32(w["max_d2"]), parallel=True, **w["kw"])
    t0 = time.perf_counter()
    knn = mk()
    t_build = time.perf_counter() - t0
    # "all the host threads it can use": the kd-tree sweep is latency-bound and was measured 3x slower
    # with every hyper-thread (128) than with one thread per core (64) on the B200 host, so probe both
    # on one iteration and give the reference the better setting
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    best = None
    for nt in sorted({ncpu, max(1, ncpu // 2)}):
        oracle.set_num_threads(nt)
        t0 = time.perf_counter()
        oracle.icp(dst, src, knn, max_iter=1, **kw)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
    oracle.set_num_threads(best[1])
    cores = best[1]
    if warmup > 0:
        oracle.icp(dst, src, knn, max_iter=warmup, **kw)
    t0 = time.perf_counter()
    if build_in_timed_region:
        knn = mk()  # SimpleICP::estimate() builds the kd-tree lazily inside the first iteration
    r = oracle.icp(dst, src, knn, max_iter=steps, **kw)
    dt = time.perf_counter() - t0
    return dict(kind=kind, cores=cores, seconds=dt, build_s=t_build, iters=r["iterations"], t_knn_s=r["t_knn_s"],
                t_est_s=r["t_est_s"], T=r["T"], num_corr=r["num_corr"])


def pick_workload(args):
    """(workload name, scaling) of this invocation: see the module docstring."""
    if args.workload:
        name = args.workload
    else:
        name = "icp_p2p_1m" if args.gpus == 1 else "icp_combined_10m"
    scaling = args.scaling or ("weak" if args.gpus == 1 else "strong")
    return name, scaling


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name, scaling = pick_workload(args)
    w = WORKLOADS[name]
    world = args.gpus
    d = make_inputs(w, 0, world, scaling)
    dst, src, nrm = d["dst"], d["src"], d["nrm"]
    # bounded sample: rank 0's shard of the same workload (its queries into the full destination cloud)
    r = cpu_reference_run(w, args.steps, args.warmup, dst, src, nrm, build_in_timed_region=True)
    its = r["iters"] / r["seconds"]
    value = its * src.shape[0]
    line = {
        "impl": "reference",
        "metric": "icp_correspondences_per_sec", "value": value, "unit": "correspondences/s",
        "iterations_per_sec": its,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * r["seconds"] / max(r["iters"], 1),
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, name, w, world, scaling, src.shape[0], dst.shape[0]),
        "cpu_baseline": {
            "value": value, "unit": "correspondences/s", "cores": r["cores"], "kind": r["kind"],
            "sample": (f"{r['iters']} ICP iterations of one rank's shard ({src.shape[0]} queries into {dst.shape[0]} "
                       f"reference points), kd-tree build ({r['build_s']:.2f} s) inside the timed region; "
                       f"kNN {r['t_knn_s']:.2f} s + estimate {r['t_est_s']:.2f} s; kNN = cilantro's vendored nanoflann "
                       "compiled in place, ICP loop = Eigen-free restatement (Eigen3 absent from the image)"),
        },
        "e2e": {"value": value, "unit": "correspondences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_config(args, name, w, world, scaling, n_src_rank, n_dst):
    return {
        "workload": (f"{name}: rigid ICP, {w['metric']} metric, k=1, {n_src_rank} source points per GPU x {world} "
                     f"GPU(s) against {n_dst} destination points (uniform random in the unit cube, seed 1, "
                     f"noise +-0.001), max_distance^2={w['max_d2']:g}, fixed iteration count (tol=0), {scaling} scaling"),
        "parallelism": (f"src sharded x{world}, dst replicated, one 16-value (p2p) / 28-value all-reduce per iteration, "
                        + ("ncclAllReduce (host loop)" if os.environ.get("CB_NO_FUSED_EXCHANGE") else
                           "exchanged over NVLink peer memory by the iteration's one-warp finish kernel, which also solves "
                           "the transform on the device; iterations enqueued back to back")),
        "l2": ("NOT flushed (--no-flush experiment; inputs smaller than L2 stay resident)" if getattr(args, "no_flush", False)
               else "flushed before every timed iteration (256 MiB memset outside the CUDA-event bracket)"),
    }


def timed_estimate(icp, ctx, cdist, world, steps, warmup, flush, kw):
    """W warm-up iterations, then one estimate() of `steps` iterations bracketed by barrier + synchronize.
    Returns (result dict, ms per step = max over ranks of the summed per-iteration event times / steps, wall s)."""
    if warmup > 0:
        icp.estimate(max_iter=warmup, flush_l2=flush, **kw)
    barrier(world)
    ctx.synchronize()
    t0 = time.perf_counter()
    res = icp.estimate(max_iter=steps, flush_l2=flush, timing=1, **kw)
    ctx.synchronize()
    barrier(world)
    wall = time.perf_counter() - t0
    assert res["iterations"] == steps, (res["iterations"], steps)
    ms_total = cdist.max_over_ranks(res["gpu_ms_total"])
    return res, ms_total / steps, wall


def dump_outputs(path, res):
    """The timed estimate()'s result as its caller receives it: the transform and the counts of the last step."""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "T.npy"), np.asarray(res["T"], np.float32))
    for key in ("num_corr", "iterations", "last_delta", "converged"):
        np.save(os.path.join(path, f"{key}.npy"), np.float64(res[key]))


def t_hash(T):
    return hashlib.sha1(np.ascontiguousarray(T, np.float32).tobytes()).hexdigest()[:16]


def icp_bench(args, name, w, scaling, ctx, rank, world, local, with_e2e=True, with_cpu=True, with_survey=True,
              clocks_wanted=True, dump_dir=None):
    """The ICP legs on `ctx` (all ranks call it); rank 0 gets the JSON-able dict, the others None.
    dump_dir: where rank 0 writes the timed call's outputs (dump_outputs)."""
    from cilantro_b200 import capi, dist as cdist, synth

    flush = not args.no_flush
    d = make_inputs(w, rank, world, scaling, pinned=True)
    dst, src, nrm, T_ref, lo = d["dst"], d["src"], d["nrm"], d["T_ref"], d["lo"]
    n_src, n_dst, n_total = src.shape[0], dst.shape[0], d["n_total"]
    n_src_all = n_total if scaling == "strong" else n_src * world
    max_d2 = np.float32(w["max_d2"])
    kw = dict(metric=w["metric"], tol=0.0, max_d2=max_d2, **w["kw"])

    # ---- value: inputs already resident in HBM, index built ------------------------------------------
    d_dst = capi.Cloud(ctx, dst, nrm)
    d_src = capi.Cloud(ctx, src, None, index_offset=lo)
    gi = d_dst.grid_info()
    d_src.grid_info()
    icp = capi.Icp(ctx, d_dst, d_src)
    sampler = ClockSampler(local)
    if rank == 0 and clocks_wanted:
        sampler.start()
    res, ms_per_step, wall = timed_estimate(icp, ctx, cdist, world, args.steps, args.warmup, flush, kw)
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, res)
    launches = res["kernel_launches"]  # this library's kernels launched by the timed estimate() call (not the warm-up)
    iter_ms = np.array([cdist.max_over_ranks(x) for x in res["iter_ms"]])
    clocks = None
    if clocks_wanted:
        # nvidia-smi needs ~0.1 s before its first sample and the legs above take milliseconds: keep the same
        # kernels running until rank 0 holds at least 3 samples taken under this load (or 3 s have passed)
        t_load = time.perf_counter()
        while True:
            need = 1.0 if (rank == 0 and len(sampler.lines) < 3 and time.perf_counter() - t_load < 3.0) else 0.0
            if cdist.max_over_ranks(need) == 0.0:
                break
            icp.estimate(max_iter=max(args.steps, 100), flush_l2=False, timing=0, **kw)
        if rank == 0:
            clocks = sampler.stop()
    its = 1e3 / ms_per_step
    value = its * n_src_all
    err = synth.frobenius(res["T"], T_ref)

    # ---- parity, part 1 (all ranks): bit-identical transforms on every rank --------------------------------
    hashes = [t_hash(res["T"])]
    if world > 1:
        import torch.distributed as dist

        box = [None] * world
        dist.all_gather_object(box, hashes[0])
        hashes = box
    rank_identical = len(set(hashes)) == 1
    assert rank_identical, f"ranks hold different transforms: {hashes}"
    # the same iteration count as the CPU arm below, on all ranks (the iteration contains a collective)
    cb_steps = 2 if w["n"] >= 1_000_000 else 3
    res_cb = icp.estimate(max_iter=cb_steps, flush_l2=False, timing=0, **kw)

    # ---- survey pose (SURVEY 8d's fixed 0.02 rad pose: outside ICP's basin at these densities, both arms stall;
    #      a valid workload all the same - every iteration keeps moving the estimate) ---------------------------
    survey = None
    if with_survey:
        ds = make_inputs(w, rank, world, scaling, survey_pose=True)
        s_src = capi.Cloud(ctx, ds["src"], None, index_offset=ds["lo"])
        s_src.grid_info()
        s_icp = capi.Icp(ctx, d_dst, s_src)
        s_res, s_ms, _ = timed_estimate(s_icp, ctx, cdist, world, args.steps, args.warmup, flush, kw)
        s_iter = np.array([cdist.max_over_ranks(x) for x in s_res["iter_ms"]])
        survey = {"ms_per_step": s_ms, "value": 1e3 / s_ms * n_src_all, "unit": "correspondences/s",
                  "iter_ms_first_last": [float(s_iter[0]), float(s_iter[-1])],
                  "transform_error_vs_generating_pose": synth.frobenius(s_res["T"], ds["T_ref"]),
                  "num_corr": s_res["num_corr"],
                  "pose": "AngleAxis(0.02 rad, (1,1,1)/sqrt 3), t = (0.01,-0.005,0.008) (SURVEY 8d)"}
        s_icp.close()
        s_src.close()

    # ---- e2e: host buffers -> upload -> index build -> full estimate() -> transform back -----------
    e2e = None
    if with_e2e:
        e2e_iters = w["iters"]
        e2e_runs = 3
        barrier(world)
        e2e_t = []
        from cilantro_b200.dist import shard_bounds

        dlo, dhi = shard_bounds(n_dst, rank, world)  # this rank's block of the replicated destination cloud
        if world > 1:
            # check, outside the timed region, that the block-wise replication gives every rank the whole cloud bit for bit
            chk = capi.Cloud.replicated(ctx, dst[dlo:dhi], nrm[dlo:dhi] if nrm is not None else None, dlo, n_dst)
            got_p, got_n = chk.download(normals=True) if nrm is not None else (chk.download(), None)
            assert np.array_equal(got_p.view(np.uint32), dst.view(np.uint32)), "replicated destination cloud differs"
            assert nrm is None or np.array_equal(got_n.view(np.uint32), nrm.view(np.uint32)), "replicated normals differ"
            chk.close()
        for _ in range(e2e_runs):
            ctx.synchronize()
            barrier(world)
            t0 = time.perf_counter()
            # what the ICP constructor of the shims does: both clouds in one call (the second upload overlaps the
            # first grid build), then the ICP object (means)
            if world == 1:
                c_dst, c_src = capi.cloud_pair(ctx, dst, nrm, src, None, offset_b=lo)
            else:
                # every rank uploads ITS block of the destination cloud; the blocks are exchanged over NVLink
                c_dst = capi.Cloud.replicated(ctx, dst[dlo:dhi], nrm[dlo:dhi] if nrm is not None else None, dlo, n_dst)
                c_src = capi.Cloud(ctx, src, None, index_offset=lo)
                c_dst.grid_info()
                c_src.grid_info()
            t2 = time.perf_counter()
            c_icp = capi.Icp(ctx, c_dst, c_src)
            t3 = time.perf_counter()
            r2 = c_icp.estimate(max_iter=e2e_iters, timing=0, **kw)  # production settings: no event instrumentation
            T_host = np.array(r2["T"])  # result read back on the host
            ctx.synchronize()
            t4 = time.perf_counter()
            barrier(world)
            e2e_t.append(time.perf_counter() - t0)
            if rank == 0:
                print(f"[e2e {name}] uploads + grid builds {1e3 * (t2 - t0):.2f} ms, icp_create {1e3 * (t3 - t2):.2f} ms, "
                      f"estimate({e2e_iters}) {1e3 * (t4 - t3):.2f} ms", file=sys.stderr)
            c_icp.close(); c_src.close(); c_dst.close()
        e2e_s = cdist.max_over_ranks(min(e2e_t))
        e2e_its = e2e_iters / e2e_s
        dst_up = dst.nbytes + (nrm.nbytes if nrm is not None else 0)
        h2d = (dst_up * (dhi - dlo) / max(n_dst, 1) + src.nbytes) / e2e_iters  # per rank
        d2h = (48 + 64) / e2e_iters  # the transform + the loop state summary, once per call
        e2e = {"value": e2e_its * n_src_all, "unit": "correspondences/s", "iterations_per_sec": e2e_its,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "what": ((f"cb_cloud_create_pair from pinned host buffers (2 uploads + 2 grid builds)" if world == 1 else
                         f"cb_cloud_create_replicated (each rank uploads 1/{world} of the destination cloud, blocks exchanged "
                         f"over NVLink) + cb_cloud_create (source shard) + 2 grid builds") + " + cb_icp_create + "
                        f"cb_icp_estimate({e2e_iters} iterations, enqueued back to back, transform kept on the device) + "
                        f"result on host; best of {e2e_runs}; {e2e_s * 1e3:.2f} ms per call")}

    # ---- parity, part 2 (N > 1): the sharded run against a single-GPU run of the whole problem on rank 0 --------
    sharded_vs_single = None
    if world > 1:
        barrier(world)
        if rank == 0:
            ctx1 = capi.Context(local)
            a_dst = capi.Cloud(ctx1, dst, nrm)
            a_src = capi.Cloud(ctx1, d["src_all"], None)
            r1 = capi.Icp(ctx1, a_dst, a_src).estimate(max_iter=args.steps, timing=0, **kw)
            sharded_vs_single = {"frob": synth.frobenius(res["T"], r1["T"]),
                                 "num_corr_equal": bool(res["num_corr"] == r1["num_corr"])}
            ctx1.close()
        barrier(world)

    if rank != 0:
        return None
    # ---- roofline of the iteration's kernels (cached pass + search / finish kernel; icp_loop.cu) --------------
    peak, peak_src = load_peaks()
    # algorithmic bytes per iteration and rank (DESIGN.md): 16 B query read per source point, every cell-sorted
    # reference point read once (16 B), + one 16 B normal gather per correspondence for the plane term
    algo_bytes = 16 * n_src + 16 * n_dst + (16 * n_src if w["metric"] == "combined" else 0)
    cold_ms = float(iter_ms[0])
    warm_ms = float(np.median(iter_ms[min(3, len(iter_ms) - 1):]))

    def frac(ms):
        a = algo_bytes / (ms * 1e-3) / 1e9
        return {"achieved": a, "frac": a / peak, "ms": ms}

    mean = frac(ms_per_step)
    tr = load_traffic(name) or {}
    roofline = {"bound": "hbm", "achieved": mean["achieved"], "peak": peak, "unit": "GB/s", "frac": mean["frac"],
                # DRAM bytes of one converged iteration's kernels (cached pass + search + finish), ncu --set full
                "traffic": (tr.get("converged_iteration") or {}).get("total") if world == 1 else None,
                "traffic_detail": tr if world == 1 else None,
                "kernel": ("one ICP iteration = icp_cached_pipe_kernel<%s> (exact re-use of the previous matches) + "
                           "icp_search_kernel<%s> (grid 1-NN of the remaining queries, grid reduction) + "
                           "icp_finish_kernel (one warp: exchange over NVLink, solve); the first iteration of a call is "
                           "icp_search_kernel + icp_finish_kernel alone" % (w["metric"], w["metric"])),
                "kernel_ms": ms_per_step, "algorithmic_bytes": algo_bytes, "peak_source": peak_src,
                "first_iteration": frac(cold_ms), "converged_iterations": frac(warm_ms),
                "iter_ms": [float(x) for x in iter_ms]}

    # ---- CPU baseline + parity on rank 0's host cores, bounded sample ----------------------------------------
    cpu = None
    parity = {"rank_identical_transforms": rank_identical, "transform_hashes": sorted(set(hashes))}
    if sharded_vs_single is not None:
        parity["sharded_vs_single_gpu"] = sharded_vs_single
    if with_cpu:
        # the CPU arm solves the GLOBAL problem (all source points) so that its transform is comparable
        src_cpu = d["src_all"] if world > 1 else src
        r = cpu_reference_run(w, cb_steps, 0, dst, src_cpu, nrm, build_in_timed_region=False)
        cits = r["iters"] / r["seconds"]
        cpu = {"value": cits * src_cpu.shape[0], "unit": "correspondences/s", "iterations_per_sec": cits, "cores": r["cores"],
               "kind": r["kind"],
               "sample": (f"{r['iters']} ICP iterations ({src_cpu.shape[0]} queries into {n_dst} reference points), "
                          f"kd-tree prebuilt (build {r['build_s']:.2f} s, 1 thread, not counted); kNN {r['t_knn_s']:.2f} s "
                          f"+ estimate {r['t_est_s']:.2f} s")}
        parity.update({
            "iterations_compared": cb_steps,
            "transform_frob_vs_cpu_arm": synth.frobenius(res_cb["T"], r["T"]),
            "num_corr_equal": bool(int(res_cb["num_corr"]) == int(r["num_corr"])),
            "num_corr": [int(res_cb["num_corr"]), int(r["num_corr"])],
        })
    out = {
        "value": value, "unit": "correspondences/s", "iterations_per_sec": its, "ms_per_step": ms_per_step,
        "config": workload_config(args, name, w, world, scaling, n_src, n_dst),
        "grid": gi,
        "transform_error_vs_generating_pose": err,
        "wall_ms_per_step_incl_flush": 1e3 * wall / args.steps,
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity": parity,
        "survey_pose": survey,
    }
    icp.close()
    d_src.close()
    d_dst.close()
    return out


def run_ours(args):
    import torch

    from cilantro_b200 import capi, dist as cdist

    rank, world, local = cdist.init_process_group()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: cilantro_b200 has no CPU fallback")
    capi.lib()
    ctx = capi.Context(local)
    cdist.attach_comm(ctx)
    name, scaling = pick_workload(args)
    w = WORKLOADS[name]
    main = icp_bench(args, name, w, scaling, ctx, rank, world, local, with_cpu=not args.no_cpu_baseline,
                     dump_dir=args.dump_outputs)

    # ---- secondary workloads ------------------------------------------------------------------------------------
    secondary = {}
    if not args.no_secondary:
        import bench_aux

        if world == 1:
            if name != "icp_combined_10m":
                sub = argparse.Namespace(**vars(args))
                sub.steps, sub.warmup = WORKLOADS["icp_combined_10m"]["iters"], 3
                r = icp_bench(sub, "icp_combined_10m", WORKLOADS["icp_combined_10m"], "weak", ctx, rank, world, local,
                              with_cpu=not args.no_cpu_baseline, clocks_wanted=False)
                r["steps"], r["warmup"] = sub.steps, sub.warmup
                secondary["icp_combined_10m"] = r
            aux = argparse.Namespace(**vars(args))
            for key, fn, steps in (("kmeans_50m", bench_aux.kmeans, 5), ("ransac_5m", bench_aux.ransac, 3),
                                   ("pca_50m", bench_aux.pca, 5)):
                aux.steps, aux.warmup = steps, 1
                try:
                    secondary[key] = bench_aux.brief(fn(aux, ctx=ctx))
                except Exception as e:  # a secondary workload must not take the headline down with it
                    secondary[key] = {"error": f"{type(e).__name__}: {e}"}
        else:
            aux = argparse.Namespace(**vars(args))
            aux.steps, aux.warmup = 5, 1
            try:
                r = bench_aux.kmeans(aux, ctx=ctx, rank=rank, world=world)
                if rank == 0:
                    secondary["kmeans_50m"] = bench_aux.brief(r)
            except Exception as e:
                secondary["kmeans_50m"] = {"error": f"{type(e).__name__}: {e}"}
    if rank != 0:
        return 0
    line = {
        "metric": "icp_correspondences_per_sec", "value": main["value"], "unit": "correspondences/s",
        "iterations_per_sec": main["iterations_per_sec"],
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
    }
    for k in ("config", "grid", "transform_error_vs_generating_pose", "wall_ms_per_step_incl_flush", "clocks", "e2e",
              "gpu_launches", "roofline", "cpu_baseline", "parity", "survey_pose"):
        line[k] = main[k]
    line["secondary"] = secondary
    print(json.dumps(line))
    return 0


def barrier(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    from bench_aux import AUX

    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS) + sorted(AUX))
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="default: weak at --gpus 1 (one shard), strong (BASELINE config 3) at --gpus N > 1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the `secondary` block (other BASELINE configs)")
    ap.add_argument("--no-flush", action="store_true",
                    help="experiments only: skip the L2 flush between timed iterations (the reported config says so)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed ICP call's outputs (transform and counts of its last step) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload in AUX):
        ap.error("--dump-outputs applies to the ICP workloads of --impl ours")
    args.warmup = max(args.warmup, 0)
    if args.workload in AUX:  # secondary single-GPU workloads (k-means, RANSAC, PCA, ...) on their own: bench_aux.py
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(AUX[args.workload](args)))
        return 0
    if args.impl == "reference":
        return run_reference(args)
    try:
        return run_ours(args)
    finally:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    sys.exit(main())
