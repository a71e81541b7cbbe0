"""A/B of feature-cloud self-kNN with long lists (DGCNN with k = 40) against the FP32 path and torch, in one process.

Shapes: DGCNN's four kNN calls (C = 3, 64, 64, 128) at 32 x 2048, k = 40 and at 32 x 1024, k = 20 (config 4), then the
batch sweep B = 4, 6, 8, 16, 32 x 2048 x 64 at k = 40 that sets the batch-size rule for long lists (`tc_fills`, hg_knn.cu).
Arms, alternated round by round: hitgeom's default dispatch, hg_tune("knn_tc", 1) (FP32 tile + row select; the 3-D
kernels at C = 3), hg_tune("knn_tc", 2) (tensor-core kernel forced; sweep only) and the reference program on the same
GPU (DGCNN's knn: -2 x^T x - xx - xx^T, then torch.topk; FP32 matmul, TF32 off).  CUDA events around `--calls` calls,
median over `--rounds` rounds, after a warm-up of every arm.  The inputs (at most 32 MB) stay L2-resident between
calls, as a DGCNN layer's input does.  Indices: every hitgeom arm equals the oracle on two sampled clouds and the other
hitgeom arms on the whole batch.  Prints the GPU name, power limit and max SM clock, then one JSON line per shape.

    python tools/knn_long_lists_ab.py [--rounds 7] [--calls 10] [--sections dgcnn40,dgcnn20,sweep] [--out DIR]

--sections dgcnn20 runs only the k = 20 shapes, which a build without long lists can run too (for a same-session
comparison with it).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "hit-adv_b200")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from hitgeom import functional as F  # noqa: E402
from hitgeom._lib import lib  # noqa: E402
from oracle import oracle as O  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=%d" % torch.cuda.current_device(),
                              "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        out = "nvidia-smi failed: %s" % e
    return out


def tune(v):
    assert lib().hg_tune(b"knn_tc", int(v)) == 0


def hitgeom_arm(knob):
    def run(pc, x, k):
        tune(knob)
        try:
            return F.knn_self(pc, k, want_vals=False)[1]
        finally:
            tune(0)
    return run


def torch_arm(pc, x, k):  # dgcnn_cls.py:7-13
    inner = -2 * torch.matmul(x.transpose(2, 1), x)
    xx = torch.sum(x ** 2, dim=1, keepdim=True)
    pairwise = -xx - inner - xx.transpose(2, 1)
    return pairwise.topk(k=k, dim=-1)[1]


def time_arm(fn, pc, x, k, calls):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        fn(pc, x, k)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / calls  # us per call


def run_shape(tag, B, N, C, k, arms, rounds, calls, seed):
    rng = np.random.default_rng(seed)
    pc_np = rng.standard_normal((B, N, C)).astype(np.float32)
    pc = torch.from_numpy(pc_np).cuda()
    x = pc.transpose(2, 1).contiguous()  # DGCNN's [B, C, N]
    fns = {name: (torch_arm if name == "torch" else hitgeom_arm(knob)) for name, knob in arms}
    outs = {}
    for name, fn in fns.items():  # warm-up, and the outputs to compare
        outs[name] = fn(pc, x, k)
    torch.cuda.synchronize()
    sample = [0, B - 1]
    _, oi = O.knn_self(pc_np[sample], k, threads=O.host_threads())
    equal = {}
    ref = None
    for name, idx in outs.items():
        if name == "torch":
            continue
        idx = idx.cpu().numpy()
        equal[name] = bool(np.array_equal(idx[sample], oi)) and (ref is None or bool(np.array_equal(idx, ref)))
        ref = idx if ref is None else ref
    times = {name: [] for name in fns}
    for _ in range(rounds):
        for name, fn in fns.items():
            times[name].append(time_arm(fn, pc, x, k, calls))
    rec = {"shape": tag, "B": B, "N": N, "C": C, "k": k,
           "us": {name: round(statistics.median(t), 1) for name, t in times.items()},
           "spread_us": {name: round(max(t) - min(t), 1) for name, t in times.items()},
           "indices_equal_oracle": equal}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--sections", default="dgcnn40,dgcnn20,sweep")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the A/B needs a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    O.build()
    info = gpu_info()
    print("# GPU (name, power limit, max SM clock): " + info, flush=True)
    recs = []
    sections = args.sections.split(",")
    layer_arms = [("default", 0), ("knn_tc=1", 1), ("torch", None)]
    for N, k in ((2048, 40), (1024, 20)):
        if "dgcnn%d" % k not in sections:
            continue
        for layer, C in enumerate((3, 64, 64, 128), start=1):
            recs.append(run_shape("dgcnn layer %d" % layer, 32, N, C, k, layer_arms, args.rounds, args.calls,
                                  1000 * layer + N + k))
    sweep_arms = [("default", 0), ("knn_tc=2", 2), ("knn_tc=1", 1)]
    for B in ((4, 6, 8, 16, 32) if "sweep" in sections else ()):
        recs.append(run_shape("batch sweep", B, 2048, 64, 40, sweep_arms, args.rounds, args.calls, 7 + B))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "knn_long_lists_ab.json"), "w") as f:
            json.dump({"gpu": info, "records": recs}, f, indent=1)


if __name__ == "__main__":
    main()
