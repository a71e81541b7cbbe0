"""A/B of the ordering states (ChamferkNNDist.temporal_seeds) against stateless calls on a MOVING cloud, in one process.

Per shape (bench.py's seeded make_clouds) and learning rate: an attack-like trajectory of `adv` -- every step adds
lr * sign(N(0, 1)) per coordinate and clips to an l_inf budget around ori -- and ChamferkNNDist fwd+bwd on it, once
stateless and once with `temporal_seeds(True)`, the two arms alternating their order step by step.  Reported per arm:
ms per step (CUDA events, counting off), orderings refit / rebuilt / built per step (hg_prune_order_counters) and the
fraction of leaf pairs the pruned passes visited (hg_prune_counters), both from a second pass over the same trajectory
with counting on; and whether loss and gradient were the same bits as the stateless arm's at every step.  Then the
sweep of the refit tolerance tau (hg_tune("prune_refit_tol", permille)) behind the default, and the refit kernel's time
with the cloud staged in shared memory or gathered from global memory (torch.profiler).  Prints one JSON line per
record, with the GPU name, power limit and max SM clock; fails without a GPU.

    python tools/order_state_ab.py [--shapes 1024x16384,2048x8192] [--lrs 1e-3,1e-2] [--steps 200]
                                   [--taus 10,25,50,100,200,400] [--out DIR]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "hit-adv_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402

from bench import make_clouds  # noqa: E402
from hitgeom import functional as F  # noqa: E402
from hitgeom._lib import lib  # noqa: E402
from hitgeom.dist_utils import ChamferkNNDist  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--id=%d" % torch.cuda.current_device(),
                          "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60, check=True).stdout.strip()
    return out


def tune(key, v):
    assert lib().hg_tune(key.encode(), int(v)) == 0


def leaf_counters():
    c = (ctypes.c_ulonglong * 4)()
    assert lib().hg_prune_counters(c) == 0
    return list(c)


def trajectory(ori, adv0, steps, lr, budget, seed=7):
    g = torch.Generator(device=ori.device).manual_seed(seed)
    adv = adv0.clone()
    for _ in range(steps):
        step = lr * torch.sign(torch.randn(adv.shape, device=adv.device, generator=g))
        adv = torch.minimum(torch.maximum(adv + step, ori - budget), ori + budget)
        yield adv


def fwd_bwd(mod, adv, ori):
    a = adv.detach().clone().requires_grad_(True)
    loss = mod(a, ori)
    loss.backward()
    return loss.detach(), a.grad


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), out


def counted_pass(mod, ori, adv0, steps, lr, budget):
    """Same trajectory with counting on: orderings per step and visited leaf-pair fractions (not timed)."""
    tune("prune_count", 1)
    F.prune_order_counters()
    leaf_counters()
    for adv in trajectory(ori, adv0, steps, lr, budget):
        fwd_bwd(mod, adv, ori)
    o = F.prune_order_counters()
    c = leaf_counters()
    tune("prune_count", 0)
    return {"refit_kept_per_step": o[0] / steps, "rebuilt_per_step": o[1] / steps, "built_per_step": o[2] / steps,
            "visited_fraction": {"chamfer": c[0] / max(c[1], 1), "knn": c[2] / max(c[3], 1)}}


def ab(B, N, ori, adv0, steps, lr, budget):
    arms = {"stateless": ChamferkNNDist(), "state": ChamferkNNDist().temporal_seeds(True)}
    for name, mod in arms.items():  # warm-up (the state arm's first call builds), then restart the trajectory
        fwd_bwd(mod, adv0, ori)
    arms["state"].temporal_seeds(True)
    ms = {k: [] for k in arms}
    same, losses = True, []
    for t, adv in enumerate(trajectory(ori, adv0, steps, lr, budget)):
        order = ("stateless", "state") if t % 2 == 0 else ("state", "stateless")
        res = {}
        for name in order:
            dt, res[name] = timed(lambda: fwd_bwd(arms[name], adv, ori))  # noqa: B023
            ms[name].append(dt)
        same &= torch.equal(res["state"][0], res["stateless"][0]) and torch.equal(res["state"][1], res["stateless"][1])
        losses.append(res["stateless"][0].clone())
    rec = {"B": B, "N": N, "lr": lr, "budget": budget, "steps": steps, "same_bits_every_step": bool(same)}
    for name in arms:
        v = ms[name]
        rec[name] = {"ms_per_step": sum(v) / len(v), "ms_median": sorted(v)[len(v) // 2], "ms_max": max(v)}
    arms["state"].temporal_seeds(True)
    for name, mod in arms.items():
        rec[name].update(counted_pass(mod, ori, adv0, steps, lr, budget))
    rec["speedup"] = rec["stateless"]["ms_per_step"] / rec["state"]["ms_per_step"]
    return rec, torch.stack(losses)


def tau_sweep(B, N, ori, adv0, steps, lr, budget, taus, ref_losses):
    rows = []
    for tau in taus:
        tune("prune_refit_tol", tau)
        mod = ChamferkNNDist().temporal_seeds(True)
        fwd_bwd(mod, adv0, ori)
        mod.temporal_seeds(True)
        v, same = [], True
        for t, adv in enumerate(trajectory(ori, adv0, steps, lr, budget)):
            dt, (loss, _) = timed(lambda: fwd_bwd(mod, adv, ori))  # noqa: B023
            v.append(dt)
            same &= torch.equal(loss, ref_losses[t])
        mod.temporal_seeds(True)
        row = {"tau_permille": tau, "ms_per_step": sum(v) / len(v), "loss_same_bits_every_step": bool(same)}
        row.update(counted_pass(mod, ori, adv0, steps, lr, budget))
        rows.append(row)
    tune("prune_refit_tol", 0)
    return {"B": B, "N": N, "lr": lr, "budget": budget, "steps": steps, "tau_sweep": rows}


def refit_kernel_times(ori, adv0, reps=5):
    """Device time of prune_refit_kernel per step (3 refits), staged in shared memory against gathered from L2."""
    from torch.profiler import ProfilerActivity, profile

    out = {}
    for stage, name in ((1, "shared_memory"), (2, "global_l2")):
        tune("prune_refit_stage", stage)
        mod = ChamferkNNDist().temporal_seeds(True)
        for _ in range(2):
            fwd_bwd(mod, adv0, ori)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                fwd_bwd(mod, adv0, ori)
            torch.cuda.synchronize()
        k = {}
        for e in prof.key_averages():
            dt = getattr(e, "device_time_total", None)
            if dt is None:
                dt = e.cuda_time_total
            for kn in ("prune_refit_kernel", "prune_order_kernel", "prune_search_kernel"):
                if kn in e.key:
                    k[kn] = k.get(kn, 0.0) + dt / 1e3 / reps
        out[name] = {kk + "_ms_per_step": v for kk, v in k.items()}
    tune("prune_refit_stage", 0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="1024x16384,2048x8192")
    ap.add_argument("--lrs", default="1e-3,1e-2")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--budget", type=float, default=0.18, help="l_inf budget around ori")
    ap.add_argument("--taus", default="10,25,50,100,200,400", help="refit tolerances [permille] of the sweep")
    ap.add_argument("--sweep-shape", default="1024x16384")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("order_state_ab.py measures on a CUDA GPU; none is available")
    recs = [{"gpu": gpu_info()}]
    print(json.dumps(recs[0]), flush=True)
    lrs = [float(v) for v in a.lrs.split(",")]
    taus = [int(v) for v in a.taus.split(",") if v]
    for s in a.shapes.split(","):
        B, N = (int(v) for v in s.split("x"))
        ori_np, adv_np = make_clouds(B, N, 1234)
        ori, adv0 = torch.from_numpy(ori_np).cuda(), torch.from_numpy(adv_np).cuda()
        for lr in lrs:
            rec, losses = ab(B, N, ori, adv0, a.steps, lr, a.budget)
            print(json.dumps(rec), flush=True)
            recs.append(rec)
            if s == a.sweep_shape and taus:
                rec = tau_sweep(B, N, ori, adv0, a.steps, lr, a.budget, taus, losses)
                print(json.dumps(rec), flush=True)
                recs.append(rec)
        if s == a.sweep_shape:
            rec = {"B": B, "N": N, "refit_gather": refit_kernel_times(ori, adv0)}
            print(json.dumps(rec), flush=True)
            recs.append(rec)
        del ori, adv0
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "order_state_ab.json"), "w") as f:
            json.dump(recs, f, indent=1)


if __name__ == "__main__":
    main()
