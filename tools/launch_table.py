"""Per-kernel device time of bench.py's default step (ChamferkNNDist fwd+bwd, make_clouds(B, N, 1234)) under
torch.profiler, in the table format kept under profiles/ (tools/launch_summary.py).

usage: python tools/launch_table.py [--clouds 1024] [--points 16384] [--steps 2] "header line" ... > profiles/rNN_x.txt
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "hit-adv_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from bench import make_clouds  # noqa: E402
from hitgeom.dist_utils import ChamferkNNDist  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--clouds", type=int, default=1024)
ap.add_argument("--points", type=int, default=16384)
ap.add_argument("--steps", type=int, default=2)
ap.add_argument("header", nargs="*")
a = ap.parse_args()
ori_np, adv_np = make_clouds(a.clouds, a.points, 1234)
ori, adv0 = torch.from_numpy(ori_np).cuda(), torch.from_numpy(adv_np).cuda()
dist = ChamferkNNDist()


def step():
    adv = adv0.clone().requires_grad_(True)
    dist(adv, ori).backward()


for _ in range(2):
    step()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(a.steps):
        step()
    torch.cuda.synchronize()
rows = []
for e in prof.key_averages():
    t = getattr(e, "device_time_total", None)
    t = e.cuda_time_total if t is None else t
    if t > 0 and e.count > 0:
        name = e.key.replace("(anonymous namespace)", "<unnamed>")
        rows.append((name.split("(")[0], e.count, t))
tot = sum(r[2] for r in rows)
for line in a.header:
    print(f"# {line}")
print(f"# total device time over {sum(r[1] for r in rows)} launches: {tot / 1e3:.2f} ms\n")
print(f"{'kernel':70s} {'launches':>8s} {'total_us':>12s} {'avg_us':>10s} {'share':>7s}")
for n, c, t in sorted(rows, key=lambda r: -r[2]):
    print(f"{n[:70]:70s} {c:8d} {t:12.1f} {t / c:10.1f} {100 * t / tot:6.2f}%")
