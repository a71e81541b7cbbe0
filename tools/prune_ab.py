"""A/B of the pruned Chamfer / self-kNN passes (hg_prune.cu) against the all-pairs kernels, in one process.

Per shape (bench.py's seeded make_clouds): hg_nn_bidir_f32 and hg_knn_self_f32 (k+1 = 6) timed with CUDA events,
pruning off and on alternately; the ordering build on its own (torch.profiler, prune_order_kernel); the fraction of
leaf pairs (32 x 32 point pairs each) the pruned passes visited, from their culling decisions; bit equality of every
output over the whole batch; the self-kNN search's drains (leaves drained, candidates inserted and warp rounds, from
hg_prune_drain_counters).  Prints one JSON line per shape with the GPU name and power limit.

    python tools/prune_ab.py [--shapes 1024x16384,2048x8192,4096x4096] [--reps 10] [--out DIR]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "hit-adv_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402

from bench import make_clouds  # noqa: E402
from hitgeom import functional as F  # noqa: E402
from hitgeom._lib import lib  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=%d" % torch.cuda.current_device(),
                              "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        out = "nvidia-smi failed: %s" % e
    return out


def tune(key, v):
    assert lib().hg_tune(key.encode(), int(v)) == 0


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def counters():
    c = (ctypes.c_ulonglong * 4)()
    assert lib().hg_prune_counters(c) == 0
    return list(c)


def drain_counters():
    c = (ctypes.c_ulonglong * 3)()
    assert lib().hg_prune_drain_counters(c) == 0
    return list(c)


def run_shape(B, N, reps, k1):
    ori_np, adv_np = make_clouds(B, N, 1234)
    ori, adv = torch.from_numpy(ori_np).cuda(), torch.from_numpy(adv_np).cuda()
    nn = lambda: F.nn_bidir(ori, adv)  # noqa: E731
    kn = lambda: F.knn_self(adv, k1)  # noqa: E731
    outs = {}
    for mode in (0, 1):  # warm-up of both paths, and the outputs compared below
        tune("prune", mode)
        outs[mode] = [t.clone() for t in nn()] + [t.clone() for t in kn()]
    torch.cuda.synchronize()
    same = all(torch.equal(x, y) for x, y in zip(outs[0], outs[1]))
    del outs
    t = {(m, w): [] for m in (0, 1) for w in ("nn", "knn")}
    for _ in range(reps):
        for mode in (0, 1):
            tune("prune", mode)
            t[(mode, "nn")].append(timed(nn))
            t[(mode, "knn")].append(timed(kn))
    tune("prune", 1)
    tune("prune_count", 1)
    counters()
    drain_counters()
    nn()
    kn()
    c = counters()
    drains, pushes, rounds = drain_counters()
    tune("prune_count", 0)
    # ordering build on its own: kernel time from the profiler (three builds per step: ori and adv for the Chamfer
    # call, adv again for the kNN call)
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        nn()
        kn()
        torch.cuda.synchronize()
    build_us, search_us = 0.0, {}
    for e in prof.key_averages():
        dt = getattr(e, "device_time_total", None)
        if dt is None:
            dt = e.cuda_time_total
        if "prune_order_kernel" in e.key:
            build_us += dt
        if "prune_search_kernel" in e.key:
            search_us[e.key[:60]] = dt

    def stats(v):
        return {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)}

    rec = {"B": B, "N": N, "k1": k1, "reps": reps, "gpu": gpu_info(), "outputs_bit_equal_whole_batch": same,
           "nn_bidir": {"off": stats(t[(0, "nn")]), "on": stats(t[(1, "nn")])},
           "knn_self": {"off": stats(t[(0, "knn")]), "on": stats(t[(1, "knn")])},
           "ordering_build_ms_per_step_3_builds": build_us / 1e3,
           "search_kernel_ms": {k: v / 1e3 for k, v in search_us.items()},
           "leaf_pairs_visited": {"chamfer": c[0], "chamfer_total": c[1], "knn": c[2], "knn_total": c[3]},
           "leaf_pairs_visited_fraction": {"chamfer": c[0] / max(c[1], 1), "knn": c[2] / max(c[3], 1)},
           # per drained leaf: candidates inserted per lane and warp rounds; busy lanes per round (of 32)
           "knn_drains": {"drains": drains, "inserted": pushes, "rounds": rounds,
                          "inserted_per_lane_per_drain": pushes / max(32 * drains, 1),
                          "rounds_per_drain": rounds / max(drains, 1),
                          "lanes_busy_per_round": pushes / max(rounds, 1)}}
    for w in ("nn_bidir", "knn_self"):
        rec[w]["speedup"] = rec[w]["off"]["median_ms"] / rec[w]["on"]["median_ms"]
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="1024x16384,2048x8192,4096x4096")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--k1", type=int, default=6)
    ap.add_argument("--min-n", type=int, default=0, help="hg_tune('prune_min_n'): lets smaller clouds take the path")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    tune("prune_min_n", a.min_n)
    recs = []
    for s in a.shapes.split(","):
        B, N = (int(v) for v in s.split("x"))
        rec = run_shape(B, N, a.reps, a.k1)
        print(json.dumps(rec), flush=True)
        recs.append(rec)
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "prune_ab.json"), "w") as f:
            json.dump(recs, f, indent=1)


if __name__ == "__main__":
    main()
