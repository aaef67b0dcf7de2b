"""Connected-component segmentation on one GPU: ConnectedComponentExtraction3f::segment with the recipe of the
reference's examples/connected_component_extraction.cpp (radius neighbourhood, NormalsProximityEvaluator at 2 degrees,
min segment size 100, max n) on synth.segment_scene, a ground plane with floating boxes and spheres (analytic normals,
r = 2.5 x the point spacing).

One JSON line per workload:
  gpu_ms           median device time of cb_cloud_segment over --calls calls, L2 flushed before each call; the stage
                   split (neighbourhood + union, finalise) is the median of the same calls;
  yardstick_ms     median host time of the count-only cb_radius_search (sizing call: one sweep over the same cloud and
                   radius, ending in a device synchronise) in the same run, L2 flushed before each call;
  cpu_*            the serial reference loop (tests/cpp/segment_oracle.cpp) on the reference kd-tree's neighbourhoods
                   (oracle/_ref) where that library was built; --no-cpu skips it;
  parity           GPU labels / offsets / points / count equal to the CPU arm's, exactly;
  device, power_limit_w: read in the same run.
Writes nothing to the tree (the oracle is compiled into a temporary directory)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from cilantro_b200 import capi, synth  # noqa: E402

WORKLOADS = {"segment_1m": 1_000_000, "segment_5m": 5_000_000}
ANGLE = float(np.float32(2.0 * np.pi / 180.0))


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def run(ctx, name, n, calls, cpu):
    pts, nrm, r2, objects, faces = synth.segment_scene(n, seed=1)
    n = pts.shape[0]
    cloud = capi.Cloud(ctx, pts, nrm)
    kw = dict(radius2=r2, evaluator="normals", max_angle=ANGLE, min_size=100, max_size=n)
    got = capi.segment(ctx, cloud, **kw)  # warm-up: index build, module load
    ms = []
    for _ in range(calls):
        ctx.flush_l2()
        r = capi.segment(ctx, cloud, want_ms=True, **kw)
        ms.append(r[4])
        assert r[3] == got[3] and np.array_equal(r[0], got[0])
    ms = np.array(ms)
    offsets = np.zeros(n + 1, np.uint64)
    total = capi.C.c_size_t()
    yard = []
    for _ in range(calls + 1):
        ctx.flush_l2()
        t0 = time.perf_counter()
        capi._check(capi.lib().cb_radius_search(ctx.h, cloud.h, cloud.h, None, capi.C.c_float(r2), capi._p(offsets), None,
                                                None, capi.C.c_size_t(0), capi.C.byref(total)))
        yard.append((time.perf_counter() - t0) * 1e3)
    yard = yard[1:]
    out = {
        "workload": name, "n": n, "radius2": r2, "segments": got[3], "expected_segments": faces,
        "labelled_points": int(got[1][-1]), "neighbour_pairs": int(total.value),
        "gpu_ms": float(np.median(ms[:, 0])), "gpu_ms_min": float(ms[:, 0].min()), "gpu_ms_max": float(ms[:, 0].max()),
        "stage_ms": {"neighbourhood_union": float(np.median(ms[:, 1])), "finalise": float(np.median(ms[:, 2]))},
        "yardstick_ms": float(np.median(yard)), "calls": calls, "l2_flushed": True,
    }
    out["ratio_to_yardstick"] = out["gpu_ms"] / out["yardstick_ms"]
    if cpu:
        import oracle
        import segment_oracle

        oracle.build()
        knn = oracle.make_knn(pts)
        t0 = time.perf_counter()
        lists = segment_oracle.neighbour_lists(pts, 0, r2, knn)
        t1 = time.perf_counter()
        want = segment_oracle.connected_components(n, lists, normals=nrm, **{k: v for k, v in kw.items() if k != "radius2"})
        t2 = time.perf_counter()
        out.update({"cpu_neighbourhoods": knn.kind, "cpu_neighbourhoods_s": t1 - t0, "cpu_loop_s": t2 - t1,
                    "cpu_threads_neighbourhoods": oracle.num_threads(), "cpu_threads_loop": 1,
                    "parity": bool(want[3] == got[3] and all(np.array_equal(a, b) for a, b in zip(want[:3], got[:3])))})
    cloud.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--no-cpu", action="store_true")
    a = ap.parse_args()
    if a.calls < 20:
        ap.error("--calls must be >= 20")
    ctx = capi.Context(0)
    info = ctx.device_info()
    plim = power_limit()
    for name in a.workloads.split(","):
        r = run(ctx, name, WORKLOADS[name], a.calls, not a.no_cpu)
        r.update({"device": info["name"] if isinstance(info, dict) else str(info), "power_limit_w": plim})
        print(json.dumps(r), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
