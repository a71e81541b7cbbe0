"""DGCNN at large clouds: feature self-kNN, edge features and one network step, hitgeom against torch, in one process.

1. `hg_knn_self_f32` at B = 8, K in {4096, 8192, 12800, 16384}, C in {64, 128}, k in {20, 40} (section knn), and at
   B = 1, 2, 4, K in {8192, 12800}, where the batch rule of hg_knn.cu decides between the two routes (section small).  Arms: hg_tune("knn_tc", 2)
   (tensor-core kernel; per-tile column norms past 4096 points), hg_tune("knn_tc", 1) (FP32 tile + row select, up to
   12800 points), hitgeom's default dispatch, and the reference program on the same GPU (DGCNN's knn: -2 x^T x - xx -
   xx^T, then torch.topk; FP32 matmul, TF32 off).  The hitgeom arms must give the same indices.
2. Edge features at B = 8 x 16384, C = 64, k in {20, 40}: hitgeom's forward and backward against the reference's torch
   composition (gather, repeat, cat, permute) and its autograd.
3. One forward + backward of a four-layer DGCNN (edge convolutions 6 -> 64, 128 -> 64, 128 -> 128, 256 -> 256) at
   B = 8 x 16384, k in {20, 40}: over model_seams against the reference's torch program.

CUDA events around `--calls` calls, median over `--rounds` rounds, arms alternated round by round after a warm-up of
every arm.  Prints the GPU name, power limit and max SM clock, then one JSON line per shape.

    python tools/dgcnn_large.py [--rounds 5] [--calls 3] [--sections knn,small,edge,net] [--out DIR]
"""
import argparse
import itertools
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "hit-adv_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402

from hitgeom import functional as F  # noqa: E402
from hitgeom import model_seams  # noqa: E402
from hitgeom._lib import lib  # noqa: E402
from oracle import torch_port as tp  # noqa: E402


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


def knn_arm(knob):
    def run(pc, x, k):
        tune(knob)
        try:
            return F.knn_self(pc, k, want_vals=False)[1]
        finally:
            tune(0)
    return run


def torch_knn(x, k):  # dgcnn_cls.py:7-13
    inner = -2 * torch.matmul(x.transpose(2, 1), x)
    xx = torch.sum(x ** 2, dim=1, keepdim=True)
    pairwise = -xx - inner - xx.transpose(2, 1)
    return pairwise.topk(k=k, dim=-1)[1]


def time_fn(fn, calls):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / calls  # us per call


def measure(fns, rounds, calls):
    for fn in fns.values():  # warm-up
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name in fns}
    for _ in range(rounds):
        for name, fn in fns.items():
            times[name].append(time_fn(fn, calls))
    return ({name: round(statistics.median(t), 1) for name, t in times.items()},
            {name: round(max(t) - min(t), 1) for name, t in times.items()})


def knn_section(rounds, calls, batches, sizes):
    recs = []
    for B, C, k, K in itertools.product(batches, (64, 128), (20, 40), sizes):
        g = torch.Generator(device="cuda").manual_seed(K + C + k)
        pc = torch.randn(B, K, C, generator=g, device="cuda")
        x = pc.transpose(2, 1).contiguous()
        arms = {"knn_tc=2": 2, "default": 0}
        if K <= 12800:
            arms["knn_tc=1"] = 1
        fns = {name: (lambda kn=kn: knn_arm(kn)(pc, x, k)) for name, kn in arms.items()}
        fns["torch"] = lambda: torch_knn(x, k)
        idx = {name: fns[name]() for name in arms}
        ref = idx["knn_tc=2"]
        equal = all(torch.equal(v, ref) for v in idx.values())
        us, spread = measure(fns, rounds, calls)
        rec = {"section": "knn", "B": B, "K": K, "C": C, "k": k, "us": us, "spread_us": spread,
               "hitgeom_arms_equal": equal}
        print(json.dumps(rec), flush=True)
        recs.append(rec)
        del pc, x, idx, ref
        torch.cuda.empty_cache()
    return recs


def edge_section(rounds, calls):
    recs = []
    B, C, N = 8, 64, 16384
    for k in (20, 40):
        g = torch.Generator(device="cuda").manual_seed(k)
        x = torch.randn(B, C, N, generator=g, device="cuda")
        idx = model_seams.knn(x, k)
        w = torch.randn(B, 2 * C, N, k, generator=g, device="cuda")
        xh, xt = x.clone().requires_grad_(), x.clone().requires_grad_()
        out_h, out_t = F.edge_feature(xh, idx), tp.get_graph_feature(xt, idx)
        equal = bool(torch.equal(out_h, out_t))
        fns = {"hitgeom fwd": lambda: F.edge_feature(x, idx),
               "torch fwd": lambda: tp.get_graph_feature(x, idx),
               "hitgeom bwd": lambda: torch.autograd.grad(out_h, xh, w, retain_graph=True),
               "torch bwd": lambda: torch.autograd.grad(out_t, xt, w, retain_graph=True)}
        us, spread = measure(fns, rounds, calls)
        rec = {"section": "edge", "B": B, "N": N, "C": C, "k": k, "us": us, "spread_us": spread,
               "forward_equal": equal}
        print(json.dumps(rec), flush=True)
        recs.append(rec)
        del out_h, out_t, xh, xt, w
        torch.cuda.empty_cache()
    return recs


class EdgeConvNet(torch.nn.Module):
    def __init__(self, k, knn, ggf):
        super().__init__()
        self.k, self.knn, self.ggf = k, knn, ggf
        g = torch.Generator().manual_seed(0)
        self.convs = torch.nn.ModuleList()
        for cin, cout in ((6, 64), (128, 64), (128, 128), (256, 256)):
            conv = torch.nn.Conv2d(cin, cout, kernel_size=1, bias=False)
            with torch.no_grad():
                conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / cin**0.5)
            self.convs.append(conv)

    def forward(self, x):
        feats = []
        for conv in self.convs:
            e = self.ggf(x, self.knn(x, self.k))
            x = torch.nn.functional.leaky_relu(conv(e), 0.2).max(dim=-1)[0]
            feats.append(x)
        return torch.cat(feats, dim=1).max(dim=-1)[0]


def net_section(rounds, calls):
    recs = []
    B, N = 8, 16384
    g = torch.Generator(device="cuda").manual_seed(1)
    pts = torch.randn(B, 3, N, generator=g, device="cuda")
    pts /= pts.abs().max()
    for k in (20, 40):
        nets = {"hitgeom": EdgeConvNet(k, model_seams.knn, lambda x, idx: model_seams.get_graph_feature(x, idx=idx)),
                "torch": EdgeConvNet(k, torch_knn, tp.get_graph_feature)}

        def step(net):
            x = pts.clone().requires_grad_()
            net(x).square().sum().backward()

        fns = {name: (lambda n=net.cuda(): step(n)) for name, net in nets.items()}
        us, spread = measure(fns, rounds, calls)
        rec = {"section": "dgcnn fwd+bwd", "B": B, "N": N, "k": k, "us": us, "spread_us": spread}
        print(json.dumps(rec), flush=True)
        recs.append(rec)
        torch.cuda.empty_cache()
    return recs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--sections", default="knn,small,edge,net")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the measurement needs a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    info = gpu_info()
    print("# GPU (name, power limit, max SM clock): " + info, flush=True)
    sections = args.sections.split(",")
    recs = []
    if "knn" in sections:
        recs += knn_section(args.rounds, args.calls, (8,), (4096, 8192, 12800, 16384))
    if "small" in sections:
        recs += knn_section(args.rounds, args.calls, (1, 2, 4), (8192, 12800))
    if "edge" in sections:
        recs += edge_section(args.rounds, args.calls)
    if "net" in sections:
        recs += net_section(args.rounds, args.calls)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "dgcnn_large.json"), "w") as f:
            json.dump({"gpu": info, "records": recs}, f, indent=1)


if __name__ == "__main__":
    main()
