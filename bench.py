#!/usr/bin/env python
"""bench.py -- point-pair distance evals/sec (fwd+bwd) of the HiT-ADV geometry hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl hitgeom|reference] [--workload c5shard|c1]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one forward+backward of the CW-kNN distance term (`ChamferkNNDist`, CW/kNN.py:104-108) over one
batch of synthetic clouds.  Default workload = BASELINE.json config 5's per-GPU shard: 1024 clouds x 16384
points per GPU (8192 clouds over 8 GPUs), Chamfer (both directions) + kNN-outlier -> 2*B*N^2 algorithmic
pair-evals per step (SURVEY.md section 8d); the backward reuses saved indices and adds none.  Weak scaling:
per-GPU work is fixed, instances are sharded, no collective on the data path.

Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.  Inputs
(402 MB per rank) exceed the 126 MB L2, so no flush is needed for c5shard; the small c1 workload flushes L2
between timed iterations.  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "hit-adv_b200"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "point-pair distance evals/sec (fwd+bwd)"
UNIT = "pair-evals/s"
FLOP_PER_PAIR = 8.0  # 4 FFMA-equivalents per pair-eval (SURVEY.md section 8d / BASELINE.md section 3)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="hitgeom", choices=["hitgeom", "reference"])
    ap.add_argument("--workload", default="c5shard", choices=["c5shard", "c1", "hitadv", "cwknn"])
    ap.add_argument("--clouds", type=int, default=0, help="clouds per GPU (default: workload's)")
    ap.add_argument("--points", type=int, default=0, help="points per cloud (default: workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-subrecords", action="store_true",
                    help="skip the c1 / hitadv / collective sub-records of the default (c5shard) line")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="CPU-baseline budget")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


C1_NAME = "C1: ChamferDist+HausdorffDist+KNNDist(k=5) fwd+bwd, 388x1024 clouds vs jittered copies"


def workload_shape(args):
    if args.workload == "c1":
        B, N = 388, 1024
        name = C1_NAME
    else:
        B, N = 1024, 16384
        name = ("C5 shard: ChamferkNNDist (Chamfer both directions + kNN-outlier k=5) fwd+bwd, "
                "1024 clouds x 16384 points per GPU (8192 clouds over 8 GPUs)")
    return (args.clouds or B), (args.points or N), name


def make_clouds(B, N, seed):
    """SURVEY.md section 8d: N(0,I) clouds, centred, max-norm 1; adv = ori + clamp(0.01 randn, +-0.05)."""
    rng = np.random.default_rng(seed)
    ori = rng.standard_normal((B, N, 3), dtype=np.float32)
    ori -= ori.mean(axis=1, keepdims=True)
    ori /= np.sqrt((ori * ori).sum(-1)).max(axis=1)[:, None, None]
    adv = ori + np.clip(0.01 * rng.standard_normal((B, N, 3), dtype=np.float32), -0.05, 0.05)
    return np.ascontiguousarray(ori, dtype=np.float32), np.ascontiguousarray(adv, dtype=np.float32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md's clocks line)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        self.mark0 = self.mark1 = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def begin(self):
        self.mark0 = time.time()

    def end(self):
        self.mark1 = time.time()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if self.mark0 is not None and self.mark0 <= t <= (self.mark1 or t) + 0.1]
        if not rows:
            rows = [r for _, r in self.rows[-3:]]
        sm, reasons, mx = [], set(), None
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------
# CPU reference arm / baseline: the reference's torch program (oracle/torch_port.py) on the host cores
# ------------------------------------------------------------------------------------------------------------
def cpu_step_fn(workload):
    from oracle import torch_port as tp

    return tp.step_cd_hd_knn if workload == "c1" else tp.step_chamfer_knn


def pairs_per_cloud(N):
    return 2.0 * N * N


def cpu_sample_plan(N, budget_s, workload):
    """How many clouds of how many points one CPU sample holds: the real N if the [N,N] FP32 matrices of the
    reference path (about a dozen live copies incl. autograd) fit in host RAM, else the largest power of two."""
    try:
        import psutil

        free = psutil.virtual_memory().available
    except Exception:
        free = 32 << 30
    n = N
    while n > 1024 and 14 * 4 * n * n > 0.5 * free:
        n //= 2
    return n


def run_cpu(workload, N, budget_s, steps=None, warmup=0):
    """Times the reference's CPU torch path on a bounded sample; returns dict(value, cores, sample, ms_per_step)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step = cpu_step_fn(workload)
    n = cpu_sample_plan(N, budget_s, workload)
    # calibrate on one small cloud to choose the clouds-per-sample
    ori, adv = make_clouds(1, min(n, 2048), 4321)
    t0 = time.time()
    step(torch.from_numpy(adv), torch.from_numpy(ori))
    rate = pairs_per_cloud(min(n, 2048)) / max(time.time() - t0, 1e-4)
    per_cloud_s = pairs_per_cloud(n) / rate
    if steps is None:
        clouds = int(max(1, min(64, budget_s / max(per_cloud_s, 1e-3))))
        steps, warmup = 1, 0
    else:
        clouds = int(max(1, min(16, (budget_s / max(steps + warmup, 1)) / max(per_cloud_s, 1e-3))))
    ori, adv = make_clouds(clouds, n, 1234)
    ori_t, adv_t = torch.from_numpy(ori), torch.from_numpy(adv)

    def one():
        """-> [(loss, grad)] of the step's calls"""
        if n >= 8192:  # one cloud at a time: the reference path needs ~1 GiB per [N,N] matrix at N=16384
            return [step(adv_t[c : c + 1], ori_t[c : c + 1]) for c in range(clouds)]
        return [step(adv_t, ori_t)]

    for _ in range(warmup):
        one()
    t0 = time.time()
    for _ in range(steps):
        out = one()
    dt = (time.time() - t0) / steps
    sample = f"{clouds} cloud(s) x {n} points per step, {steps} step(s)" + ("" if n == N else f" (N reduced from {N}: host RAM)")
    return {"value": clouds * pairs_per_cloud(n) / dt, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
            "ms_per_step": dt * 1e3,
            "outputs": {"loss": torch.stack([l.reshape(()) for l, _ in out]), "grad": torch.cat([g for _, g in out])}}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B, N, name = workload_shape(args)
    r = run_cpu(args.workload, N, budget_s=max(30.0, 12.0 * (args.steps + args.warmup)), steps=args.steps,
                warmup=args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": distance_config(args.workload, B, N, name),
            "note": "reference CPU torch path (oracle/torch_port.py restatement) on the host cores, bounded sample",
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, **r["outputs"])
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# hitgeom arm
# ------------------------------------------------------------------------------------------------------------
def traffic_table():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the hot kernels, read from the tracked profile
    summary profiles/traffic.json (written by tools/ncu_summary.py from `ncu --set full` captures)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


def oracle_parity(workload, which, ori_np, adv_np, ori_d, adv_d, grad_d):
    """Clouds `which` of the TIMED batch against the CPU oracle, outside the timed region: nearest-neighbour and kNN
    indices and values bit for bit, the step's gradient norm-wise (SURVEY.md section 8a).  The GPU side re-runs the
    full-batch calls, i.e. the very kernel instantiations the timed steps launched."""
    from hitgeom import functional as F
    from oracle import oracle as O

    B = ori_np.shape[0]
    with torch.no_grad():
        m1, a1, m2, a2 = F.nn_bidir(ori_d, adv_d.detach())
        kv, ki = F.knn_self(adv_d.detach(), 6)
    sel = torch.as_tensor(which, device=ori_d.device)
    g = {k: v[sel].cpu().numpy() for k, v in dict(m1=m1, a1=a1, m2=m2, a2=a2, kv=kv, ki=ki, grad=grad_d).items()}
    del m1, a1, m2, a2, kv, ki
    ori, adv = ori_np[which], adv_np[which]
    n = len(which)
    thr = min(n, O.host_threads())
    o1, oa1, o2, oa2 = O.nn_bidir(ori, adv, threads=thr)
    ov, oi = O.knn_self(adv, 6, threads=thr)
    _, mask, _ = O.knn_outlier_fwd(ov, 1.05)
    ones, zeros = np.ones(n, np.float32), np.zeros(n, np.float32)
    l1, l2, h1, h2 = O.set_loss(o1, o2, 0)
    cd_g = O.set_loss_bwd(ori, adv, oa1, oa2, h1, h2, ones, zeros, 0)
    kn_g = O.knn_outlier_bwd(adv, oi, mask, ones)
    if workload == "c1":
        _, _, hh1, hh2 = O.set_loss(o1, o2, 1)
        want = (cd_g + O.set_loss_bwd(ori, adv, oa1, oa2, hh1, hh2, ones, zeros, 1) + kn_g) / B
    else:
        want = (5.0 * cd_g + 3.0 * kn_g) / B
    num = np.abs(g["grad"] - want).reshape(n, -1).max(1)
    den = np.maximum(np.abs(want).reshape(n, -1).max(1), 1e-30)
    rec = {"clouds": int(n), "cloud_ids": [int(c) for c in which],
           "nn_indices_exact": bool(np.array_equal(g["a1"], oa1) and np.array_equal(g["a2"], oa2)),
           "nn_values_exact": bool(np.array_equal(g["m1"], o1) and np.array_equal(g["m2"], o2)),
           "knn_indices_exact": bool(np.array_equal(g["ki"], oi)), "knn_values_exact": bool(np.array_equal(g["kv"], ov)),
           "grad_normwise": float((num / den).max()), "grad_tolerance": 1e-5,
           "checker": "oracle/hitgeom_oracle.c (CPU restatement pinned to the reference's golden vectors)"}
    rec["indices_exact"] = rec["nn_indices_exact"] and rec["knn_indices_exact"]
    rec["ok"] = bool(rec["indices_exact"] and rec["nn_values_exact"] and rec["knn_values_exact"]
                     and rec["grad_normwise"] < 1e-5)
    return rec


def distance_record(workload, B, N, name, steps, warmup, rank, world, local, with_e2e=True, sampler_on=True):
    """Times one distance workload (config-5 shard or config 1) on this rank's GPU; returns the record dict (on every
    rank: the max-over-ranks reductions are collective)."""
    from hitgeom import _lib, sharding
    from hitgeom.dist_utils import ChamferDist, ChamferkNNDist, HausdorffDist, KNNDist

    dev = torch.device("cuda", local)
    ori_np, adv_np = make_clouds(B, N, 1234 + rank)
    ori_h = torch.from_numpy(ori_np).pin_memory()
    adv_h = torch.from_numpy(adv_np).pin_memory()
    grad_h = torch.empty_like(adv_h).pin_memory()
    ori_d = ori_h.to(dev, non_blocking=True)
    adv_d = adv_h.to(dev, non_blocking=True).requires_grad_()
    small = workload == "c1"

    def make_fwd_bwd(temporal, overlap=False):
        """temporal=True: the kNN term keeps last call's neighbour indices as seeds (what an attack loop does).
        overlap=True (config 1): the kNN term, which does not depend on the other two, is enqueued on a forked stream
        (hitgeom.overlap.side_branch) -- at 388 x 1024 no single kernel fills 148 SMs."""
        if small:
            from hitgeom.dist_utils import shared_distance_pass
            from hitgeom.overlap import side_branch

            cd, hd, kd = ChamferDist(), HausdorffDist(), KNNDist(k=5).temporal_seeds(temporal)

            def fn(zero_grad_in_place=False):
                if zero_grad_in_place:
                    adv_d.grad.zero_()
                else:
                    adv_d.grad = None
                with shared_distance_pass():  # Chamfer and Hausdorff of the same pair: one distance pass (SURVEY 8d)
                    if overlap:
                        with side_branch() as br:
                            l_knn = kd(adv_d)
                        loss = cd(adv_d, ori_d) + hd(adv_d, ori_d) + br.join(l_knn)
                    else:
                        loss = cd(adv_d, ori_d) + hd(adv_d, ori_d) + kd(adv_d)
                loss.backward()
                return loss
        else:
            dist_func = ChamferkNNDist().temporal_seeds(temporal)

            def fn(zero_grad_in_place=False):
                if zero_grad_in_place:
                    adv_d.grad.zero_()
                else:
                    adv_d.grad = None
                loss = dist_func(adv_d, ori_d)
                loss.backward()
                return loss
        return fn

    fwd_bwd = make_fwd_bwd(False, overlap=small)
    fwd_bwd_serial = make_fwd_bwd(False) if small else fwd_bwd

    pairs_step = B * pairs_per_cloud(N)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if small else None
    flush_rd = torch.zeros(64 << 20, dtype=torch.float32, device=dev) if small else None

    def l2_flush():
        if flush is not None:
            flush.zero_()   # write 256 MiB: evicts everything ...
            flush_rd.sum()  # ... then read another 256 MiB, so that the write's dirty lines are out before the timed step

    for _ in range(max(warmup, 3)):
        fwd_bwd()
    torch.cuda.synchronize()
    step, eager_ms, serial_ms = fwd_bwd, None, None
    if small:
        # config 1 is ~0.3 ms of kernel work behind ~25 launches: launch-bound.  An attack loop replays the step as a
        # CUDA graph (hitgeom.cw_knn graph=True); time that, and report the eager figure next to it.
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for s_, e_ in evs:  # the eager figure first (launch by launch, one stream: CPU-bound): informational only
            l2_flush()
            s_.record()
            fwd_bwd_serial()
            e_.record()
        torch.cuda.synchronize()
        eager_ms = sorted(s_.elapsed_time(e_) for s_, e_ in evs)[len(evs) // 2]
        # a fresh leaf (same storage) for the captured steps: its gradient accumulator is then created on the warm-up
        # side stream, not on the legacy default stream the eager warm-up above ran on (PyTorch's rule for capturing a
        # backward pass; the closures below see the rebinding)
        adv_d = adv_d.detach().requires_grad_()
        adv_d.grad = torch.zeros_like(adv_d)

        def capture(fn):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    fn(True)
            torch.cuda.current_stream().wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = fn(True)
            g.hold = (adv_d.grad, out)  # the replays write into this gradient buffer: keep it alive with the graph
            return g, out

        graph, graph_loss = capture(fwd_bwd)
        torch.cuda.synchronize()
        # the same step with the three terms on ONE stream, for the record
        graph_serial, _ = capture(fwd_bwd_serial)
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for s_, e_ in evs:
            l2_flush()
            s_.record()
            graph_serial.replay()
            e_.record()
        torch.cuda.synchronize()
        serial_ms = sum(s_.elapsed_time(e_) for s_, e_ in evs) / len(evs)
        del graph_serial

        def step():
            graph.replay()
            return graph_loss

    # ---- device-resident timing ---------------------------------------------------------------------------
    sampler = ClockSampler(local) if (rank == 0 and sampler_on) else None
    sharding.barrier()
    torch.cuda.synchronize()
    _lib.prof_enable(True)
    launches0 = _lib.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    if sampler:
        sampler.begin()
    for s, e in evs:
        l2_flush()
        s.record()
        loss_dev = step().detach()  # detached, so the step's autograd graph is freed before the next step runs
        e.record()
    torch.cuda.synchronize()
    # what the last timed step computed (config 1: the captured graph's output buffers, rewritten by any later replay)
    grad_dev = (graph.hold[0] if small else adv_d.grad).detach().clone()
    loss_dev = loss_dev.clone()
    if sampler:
        sampler.end()
    sharding.barrier()
    launches = (_lib.launch_count() - launches0) // steps
    if small:  # a graph replay re-runs the captured kernels without passing the counter: count eagerly
        l0 = _lib.launch_count()
        fwd_bwd()
        launches = _lib.launch_count() - l0
    ms_local = sum(s.elapsed_time(e) for s, e in evs) / steps
    ms = sharding.max_over_ranks(ms_local)
    if eager_ms is not None:  # the per-kernel event hooks only fire on eager launches; one stream: kernels timed alone
        _lib.prof_enable(True)
        for _ in range(steps):
            l2_flush()
            fwd_bwd_serial()
        torch.cuda.synchronize()
    nn_ms, nn_n = _lib.prof_read("nn_bidir")
    knn_ms, knn_n = _lib.prof_read("knn")
    _lib.prof_enable(False)
    clocks = sampler.stop() if sampler else {}

    # ---- the same step with temporal kNN seeds (attack-loop usage: KNNDist.temporal_seeds) -----------------------
    temporal = None
    try:
        fb_t = make_fwd_bwd(True, overlap=small)
        for _ in range(3):
            fb_t()
        if small:
            adv_d.grad = torch.zeros_like(adv_d)
            g_t, _ = capture(fb_t)
            run_t = g_t.replay
        else:
            run_t = fb_t
        torch.cuda.synchronize()
        evs_t = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for s_, e_ in evs_t:
            l2_flush()
            s_.record()
            run_t()
            e_.record()
        torch.cuda.synchronize()
        t_ms = sharding.max_over_ranks(sum(s_.elapsed_time(e_) for s_, e_ in evs_t) / steps)
        same = bool(torch.equal(adv_d.grad, grad_dev))
        temporal = {"ms_per_step": t_ms, "value": world * pairs_step / (t_ms * 1e-3), "unit": UNIT,
                    "gradient_same_bits_as_stateless": same,
                    "what": "kNN thresholds seeded from the previous call's neighbour indices (hg_knn_self_temporal_f32) "
                            "instead of the spatial pre-pass; the benchmark repeats one cloud, an attack loop moves it by "
                            "a learning-rate step per call (tools/knn_small_sweep.py: +1..5 % kernel time at 1e-3..5e-3)"}
    except Exception as e:  # noqa: BLE001
        temporal = {"error": f"{type(e).__name__}: {e}"}

    # ---- parity of the timed batch against the CPU oracle (outside the timed region, rank 0) -----------------
    parity = None
    if rank == 0:
        which = sorted({0, B // 3, (2 * B) // 3, B - 1}) if small else [0, B - 1]
        try:
            parity = oracle_parity(workload, which, ori_np, adv_np, ori_d, adv_d, grad_dev)
        except Exception as e:  # noqa: BLE001 -- reported in the line, never hidden
            parity = {"ok": False, "error": f"{type(e).__name__}: {e}"}

    # ---- end-to-end: host buffers in, gradient + loss back to the host, every step ---------------------------
    e2e = None
    if with_e2e:
        if small:
            def e2e_step():  # host buffers in, the replayed step, gradient + loss back out
                with torch.no_grad():
                    adv_d.copy_(adv_h, non_blocking=True)
                    ori_d.copy_(ori_h, non_blocking=True)
                graph.replay()
                grad_h.copy_(graph.hold[0], non_blocking=True)
                return float(graph_loss.item())
        else:
            # the C ABI's host-buffer entry point: chunks of clouds, copies on their own streams behind the kernels
            from hitgeom.host import ChamferKnnHostStep

            host_step = ChamferKnnHostStep(N, chunk_clouds=min(512, B))
            cloud_loss_h = np.empty(B, dtype=np.float32)

            def e2e_step():
                return host_step(adv_h, ori_h, grad_h, cloud_loss_out=cloud_loss_h)[0]

        e2e_loss = e2e_step()
        torch.cuda.synchronize()
        if not small:  # same kernels as the device-resident path: the gradient must be the same bits
            assert torch.equal(grad_h, grad_dev.cpu()), "host-buffer step disagrees with the device-resident step"
        sharding.barrier()
        torch.cuda.synchronize()
        evs_e = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for e0, e1 in evs_e:
            l2_flush()  # (config 1 only; outside the timed region, as for the device-resident steps)
            e0.record()
            e2e_loss = e2e_step()  # ends with the device->host read of the loss: the step is complete at e1
            e1.record()
        torch.cuda.synchronize()
        sharding.barrier()
        e2e_ms = sharding.max_over_ranks(sum(e0.elapsed_time(e1) for e0, e1 in evs_e) / steps)
        e2e = {"value": world * pairs_step / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": int(adv_h.numel() * 4 + ori_h.numel() * 4),
               "d2h_bytes_per_step": int(grad_h.numel() * 4 + (4 if small else 4 * B)), "loss": e2e_loss,
               "api": "pinned host buffers -> captured step (module calls) -> pinned host gradient + loss" if small else
                      "hg_chamfer_knn_step_host_f32 (C ABI, host buffers, chunks of up to 512 clouds, short ones at both ends: one compute stream, copies on two copy streams)"}

    pk, pk_src = peaks()
    info = _lib.device_info()
    sm_max_mhz = float(clocks.get("sm_max_mhz") or pk.get("sm_max_mhz") or info["clock_khz"] / 1e3)
    fp32_peak_tflops = info["sm_count"] * 128 * 2 * sm_max_mhz * 1e6 / 1e12
    # dominant kernel = the tagged hot kernel with the larger share of the step
    tagged = {"nn_bidir_d3_kernel": (nn_ms, nn_n, B * float(N) * N), "knn3_kernel": (knn_ms, knn_n, B * float(N) * N)}
    kname = max(tagged, key=lambda k: tagged[k][0])
    k_ms, k_n, k_pairs = tagged[kname]
    k_avg_ms = k_ms / max(k_n, 1)
    achieved = k_pairs * FLOP_PER_PAIR / (k_avg_ms * 1e-3) / 1e12 if k_avg_ms > 0 else 0.0
    alg_bytes = B * (2 * N) * 12 + B * (2 * N) * 8
    tt = traffic_table().get(f"{B}x{N}", {})
    per_kernel = {}
    for k, (t_ms, t_n, t_pairs) in tagged.items():
        avg = t_ms / max(t_n, 1)
        tf = t_pairs * FLOP_PER_PAIR / (avg * 1e-3) / 1e12 if avg > 0 else 0.0
        per_kernel[k] = {"avg_launch_ms": avg, "launches_timed": t_n, "achieved_tflops": tf,
                         "frac": tf / fp32_peak_tflops if fp32_peak_tflops else None,
                         "share_of_step": avg * (t_n / max(steps, 1)) / ms_local if ms_local > 0 else None}
    step_tflops = pairs_step * FLOP_PER_PAIR / (ms_local * 1e-3) / 1e12
    try:  # measured FFMA throughput next to the computed figure (synchronising probe, outside every timed region)
        fp32_measured = _lib.probe_fp32_peak()
    except Exception:  # noqa: BLE001
        fp32_measured = None
    roofline = {
        "bound": "fp32", "kernel": kname, "achieved": achieved, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
        "frac": achieved / fp32_peak_tflops if fp32_peak_tflops else None,
        "peak_measured": fp32_measured, "frac_of_measured_peak": achieved / fp32_measured if fp32_measured else None,
        "peak_measured_source": "hg_probe_fp32_peak: 16 independent FFMA chains per thread, 8 CTAs of 256 threads per SM, CUDA events",
        "traffic": (tt.get(kname) or {}).get("dram_bytes"), "traffic_source": (tt.get(kname) or {}).get("source"),
        "peak_source": f"computed {info['sm_count']} SMs x 128 FP32 lanes x 2 x {sm_max_mhz:.0f} MHz (no FP32 figure in MEASURED_PEAKS.json)",
        "avg_launch_ms": k_avg_ms, "launches_timed": k_n, "algorithmic_pair_evals_per_launch": k_pairs,
        "flop_per_pair_eval": FLOP_PER_PAIR, "kernels": per_kernel,
        "whole_step": {"achieved": step_tflops, "frac": step_tflops / fp32_peak_tflops if fp32_peak_tflops else None,
                       "what": "all pair-evals of the step x 8 FLOP / ms_per_step (this rank)" + (", graph replay" if small else "")},
        "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / (k_avg_ms * 1e-3) / 1e9 if k_avg_ms > 0 else 0.0,
                "peak_gbs": pk.get("hbm_gbs"), "peak_source": pk_src},
    }
    rec = {"value": world * pairs_step / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
           "config": distance_config(workload, B, N, name, eager_ms, serial_ms), "clocks": clocks, "roofline": roofline,
           "parity_check": parity, "gpu_launches": int(launches), "temporal_seeds": temporal}
    if e2e is not None:
        rec["e2e"] = e2e
    rec["_grad_dev"] = grad_dev  # handed to the collective timing (config-5-size gather), dropped from the line
    rec["_loss_dev"] = loss_dev
    return rec


def distance_config(workload, B, N, name, eager_ms=None, serial_ms=None):
    cfg = {"workload": name, "clouds_per_gpu": B, "points": N, "k": 5,
           "l2": ("L2 flushed (256 MiB write + 256 MiB read) between timed iterations" if workload == "c1" else
                  f"inputs ({B * N * 24 / 1e6:.0f} MB/rank) exceed the 126 MB L2" if B * N * 24 > 126e6 else
                  "inputs fit in L2 (not flushed)"),
           "pair_evals_per_step_per_gpu": B * pairs_per_cloud(N)}
    if workload == "c1":
        cfg["replay"] = ("step replayed as one CUDA graph; the kNN term is enqueued on a forked stream "
                         "(hitgeom.overlap.side_branch) and captured as a parallel arm of the graph")
        if eager_ms is not None:
            cfg["eager_ms_per_step"] = eager_ms
        if serial_ms is not None:
            cfg["one_stream_graph_ms_per_step"] = serial_ms
    return cfg


def gather_record(x, world, reps=3):
    """The end-of-attack collective (SURVEY.md section 8e) at this workload's size: NCCL all_gather of the per-rank
    adversarial clouds.  CUDA events on the current stream, max over ranks, best of `reps` after one warm-up."""
    from hitgeom import sharding

    n_total = x.shape[0] * world
    best, t = None, {}
    for i in range(reps + 1):
        t = {}
        sharding.barrier()
        torch.cuda.synchronize()
        out = sharding.gather_clouds(x, n_total, timing=t)
        torch.cuda.synchronize()
        ok = bool(out.shape[0] == n_total)
        del out
        if t.get("events") is not None and i > 0:
            ms = sharding.max_over_ranks(t["events"][0].elapsed_time(t["events"][1]))
            best = ms if best is None else min(best, ms)
    rec = {"op": "all_gather_into_tensor", "backend": "nccl" if world > 1 else "none (single rank: no exchange)",
           "bytes_per_rank": t.get("bytes_per_rank"), "bytes_total": t.get("bytes_total"), "ms": best, "ok": ok}
    if best:
        rec["algbw_gbs"] = t["bytes_total"] / (best * 1e-3) / 1e9
        rec["busbw_gbs"] = rec["algbw_gbs"] * (world - 1) / world
    return rec


def hitadv_record(rank, world, local, iters, warm_iters=5):
    """BASELINE config 2 sharded by instance: every rank attacks its block of 256 clouds (weak scaling) through
    `sharding.run_sharded`, which ends with the NCCL all_gather of the adversarial clouds and the all_reduce of the
    counters (util/other_utils.py:33-43,87-98).  Timed twice: the iteration launched kernel by kernel (eager), and
    replayed as one CUDA graph per iteration (`HiT_ADV(graph=True)`); `value` is the faster of the two, both are listed."""
    from hitgeom import _lib, sharding
    from hitgeom.hit_adv import HiT_ADV, UntargetedLogitsAdvLoss
    from util_models import PointNetCls

    B, K = 256, 1024
    dev = torch.device("cuda", local)
    data_all, target_all = hitadv_inputs(world * B, K, 1234)
    model = PointNetCls(40, seed=0).to(dev)
    state = {}

    def attack_block(n_iter, graph):
        def fn(data, target):
            att = HiT_ADV(model, UntargetedLogitsAdvLoss(kappa=30.0), clip_func=None, binary_step=1, num_iter=n_iter,
                          graph=graph, **HITADV_HP)
            torch.manual_seed(0)
            adv, succ = att.attack_device(data, target)
            state["att"] = att
            return adv, {"success": succ, "clouds": float(data.shape[0])}
        return fn

    lo, hi = sharding.shard_range(world * B)
    modes = {}
    for graph in (False, True):
        tag = "graph" if graph else "eager"
        n_iter = iters + CAPTURED_AFTER if graph else iters  # graph mode: `iters` replays after the eager lead-in
        try:
            attack_block(warm_iters, graph)(data_all[lo:hi], target_all[lo:hi])
            torch.cuda.synchronize()
            sharding.barrier()
            launches0 = _lib.launch_count()
            timing = {}
            t0 = time.time()
            adv_all, counters = sharding.run_sharded(attack_block(n_iter, graph), data_all, target_all, timing=timing)
            torch.cuda.synchronize()
            wall = time.time() - t0
            sharding.barrier()
            att = state["att"]
            if graph:
                it_ms = sharding.max_over_ranks(att.replay_ms / max(att.replays, 1))
            else:
                it_ms = sharding.max_over_ranks(att.loop_ms / iters)
            gather_ms = None
            if timing.get("events") is not None:
                gather_ms = sharding.max_over_ranks(timing["events"][0].elapsed_time(timing["events"][1]))
            # the same gather again, ranks aligned by a barrier first (the figure above includes the wait for the
            # slowest rank to finish its attack: arrival skew, not transfer time)
            aligned = gather_record(adv_all[lo:hi].contiguous(), world, reps=2) if world > 1 else {}
            modes[tag] = {"ms_per_iteration": it_ms, "cloud_iterations_per_s": world * B / (it_ms * 1e-3),
                          "attack_iters_per_s_per_batch": 1e3 / it_ms,
                          "iterations_timed": int(att.replays) if graph else iters,
                          "e2e_ms_per_iteration": sharding.max_over_ranks(wall * 1e3 / n_iter),
                          "hitgeom_launches_per_iteration": int((_lib.launch_count() - launches0) // iters) if not graph else None,
                          "collective": {"op": "all_gather_into_tensor", "backend": "nccl" if world > 1 else "none (single rank)",
                                         "bytes_per_rank": timing.get("bytes_per_rank"), "bytes_total": timing.get("bytes_total"),
                                         "ms_incl_arrival_skew": gather_ms, "ms": aligned.get("ms"),
                                         "busbw_gbs": aligned.get("busbw_gbs"), "gathered_clouds": int(adv_all.shape[0]),
                                         "counters_all_reduced": counters}}
        except Exception as e:  # noqa: BLE001 -- a failing mode is reported, the other one still counts
            modes[tag] = {"error": f"{type(e).__name__}: {e}"}
            try:
                torch.cuda.synchronize()
            except Exception:  # noqa: BLE001
                pass
    ok = {k: v for k, v in modes.items() if "ms_per_iteration" in v}
    if not ok:
        return {"metric": HITADV_METRIC, "value": None, "modes": modes}
    best = min(ok, key=lambda k: ok[k]["ms_per_iteration"])
    m = ok[best]
    return {"metric": HITADV_METRIC, "value": m["cloud_iterations_per_s"], "unit": "cloud-iterations/s", "mode": best,
            "attack_iters_per_s_per_batch": m["attack_iters_per_s_per_batch"], "ms_per_iteration": m["ms_per_iteration"],
            "iterations": iters, "batch_per_gpu": B, "points": K, "scaling": "weak",
            "e2e": {"value": world * B / (m["e2e_ms_per_iteration"] * 1e-3), "unit": "cloud-iterations/s",
                    "ms_per_iteration": m["e2e_ms_per_iteration"],
                    "what": "whole run_sharded call: host data in, centre selection, iterations (incl. warm-up + capture), "
                            "all_gather + all_reduce"},
            "collective": m["collective"], "modes": modes,
            "workload": f"C2: HiT-ADV attack loop (ShapeAttack/HiT_ADV.py:125-273), {B} clouds x {K} points per GPU, "
                        "random-init PointNet victim, eval.py defaults, binary_step=1",
            "note": "value = device time per inner iteration (CUDA events around the loop / the replayed iterations), max over ranks"}


DUMP_ARRAY_BYTES = 48 << 20  # per array; the largest output is the only one near it, so a directory stays under 64 MB
CAPTURED_AFTER = 3  # eager iterations HiT_ADV / CWKNN(graph=True) run before capturing one (hit_adv.py, cw_knn.py)


def dump_outputs(path, **arrays):
    """--dump-outputs: what a caller of the timed path receives from its last step, one DIR/<name>.npy per array,
    float64 if it is float64 and float32 otherwise.  An array larger than DUMP_ARRAY_BYTES is sampled by whole clouds
    (rows of its first axis), picked with a fixed seed from its shape alone, so runs with the same arguments store the
    same clouds and two builds can be compared file for file."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > DUMP_ARRAY_BYTES:
            n = max(1, DUMP_ARRAY_BYTES // (a[0].nbytes or 1))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], n, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def main_hitgeom(args):
    from hitgeom import _lib, sharding

    rank, world, local = sharding.init()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(torch.device("cuda", local))
    _lib.lib()  # fail loudly if the CUDA extension is missing
    B, N, name = workload_shape(args)
    rec = distance_record(args.workload, B, N, name, args.steps, args.warmup, rank, world, local)
    grad_dev, loss_dev = rec.pop("_grad_dev"), rec.pop("_loss_dev")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss=loss_dev, grad=grad_dev)
    line = {"metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": rec["config"], "clocks": rec["clocks"],
            "roofline": rec["roofline"], "e2e": rec["e2e"], "parity_check": rec["parity_check"],
            "gpu_launches": rec["gpu_launches"], "temporal_seeds": rec["temporal_seeds"]}
    if args.workload == "c5shard" and not args.no_subrecords:
        # the other half of BASELINE's metric and the workload its 60 % target is worded on, in the same driver-run line
        try:
            line["collective"] = gather_record(grad_dev, world)
            line["collective"]["what"] = ("end-of-attack all_gather of the adversarial clouds at config-5 size "
                                          f"([{B},{N},3] f32 per rank), sharding.gather_clouds")
        except Exception as e:  # noqa: BLE001
            line["collective"] = {"ok": False, "error": f"{type(e).__name__}: {e}"}
        del grad_dev
        torch.cuda.empty_cache()
        try:
            c1 = distance_record("c1", 388, 1024, C1_NAME, args.steps, args.warmup, rank, world, local,
                                 sampler_on=False)
            c1.pop("_grad_dev")
            c1.pop("_loss_dev")
            line["c1"] = c1
        except Exception as e:  # noqa: BLE001
            line["c1"] = {"ok": False, "error": f"{type(e).__name__}: {e}"}
        torch.cuda.empty_cache()
        try:
            line["hitadv"] = hitadv_record(rank, world, local, iters=args.steps)
        except Exception as e:  # noqa: BLE001
            line["hitadv"] = {"ok": False, "error": f"{type(e).__name__}: {e}"}
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    if world == 1 and not args.no_cpu_baseline:
        try:
            r = run_cpu(args.workload, N, args.cpu_seconds, steps=args.steps)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as e:  # the baseline must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# BASELINE config 2: the HiT-ADV attack loop on 1024-point clouds against a random-init PointNet (eval.py defaults:
# batch 256, central_num 192, total_central_num 256, curv_loss_knn 16, budget 0.55, cd/ker/hide = 1e-4/1/1, kappa 30)
# A "step" = one inner attack iteration over the batch (deformation -> victim fwd/bwd -> losses -> Adam ->
# best-result bookkeeping).  value = cloud-iterations per second.
# ------------------------------------------------------------------------------------------------------------
HITADV_METRIC = "HiT-ADV attack cloud-iterations/sec"
HITADV_HP = dict(attack_lr=1e-2, init_weight=10.0, max_weight=80.0, cd_weight=1e-4, curv_weight=0, ker_weight=1.0,
                 hide_weight=1.0, curv_loss_knn=16, central_num=192, total_central_num=256, max_sigm=1.2, min_sigm=0.1,
                 budget=0.55, alpha=1)


def hitadv_inputs(B, K, seed):
    ori, _ = make_clouds(B, K, seed)
    rng = np.random.default_rng(seed + 1)
    nrm = rng.standard_normal((B, K, 3)).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    data = torch.from_numpy(np.concatenate([ori, nrm], axis=-1))
    target = torch.from_numpy(rng.integers(0, 40, B))
    return data, target


def hitadv_cpu(B, K, iters):
    """The reference loop (oracle/hitadv_port.py, bit-identical to the reference class here) on the host cores."""
    from oracle import hitadv_port as hp
    from util_models import PointNetCls

    torch.set_num_threads(os.cpu_count() or 1)
    data, target = hitadv_inputs(B, K, 4321)
    model = PointNetCls(40, seed=0)
    torch.manual_seed(0)
    t0 = time.time()
    adv, succ, _ = hp.attack(model, data, target, dict(HITADV_HP, kappa=30.0, binary_step=1, num_iter=iters))
    dt = time.time() - t0
    return {"value": B * iters / dt, "unit": "cloud-iterations/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"batch of {B} clouds x {K} points, {iters} iterations (incl. one-off setup)", "ms_per_step": dt / iters * 1e3,
            "outputs": {"adv": adv, "success": np.float64(succ)}}


def main_hitadv(args):
    from util_models import PointNetCls

    B, K = (args.clouds or 256), (args.points or 1024)
    name = f"C2: HiT-ADV attack loop, batch {B} x {K} points, random-init PointNet victim, eval.py defaults"
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return
        r = hitadv_cpu(8, K, args.steps)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, **r["outputs"])
        line = {"impl": "reference", "metric": HITADV_METRIC, "value": r["value"], "unit": r["unit"], "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": name},
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": r["value"], "unit": r["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return
    from hitgeom import _lib, sharding
    from hitgeom.hit_adv import HiT_ADV, UntargetedLogitsAdvLoss

    rank, world, local = sharding.init()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    data, target = hitadv_inputs(B, K, 1234 + rank)
    model = PointNetCls(40, seed=0).to(dev)
    steps = args.steps

    def run(n_iter):
        att = HiT_ADV(model, UntargetedLogitsAdvLoss(kappa=30.0), clip_func=None, binary_step=1, num_iter=n_iter, **HITADV_HP)
        torch.manual_seed(0)
        t0 = time.time()
        adv, succ = att.attack(data, target)
        torch.cuda.synchronize()
        return att, time.time() - t0, {"adv": adv, "success": np.float64(succ)}

    run(max(5, args.warmup))
    sampler = ClockSampler(local) if rank == 0 else None
    sharding.barrier()
    launches0 = _lib.launch_count()
    if sampler:
        sampler.begin()
    att, wall, out = run(steps)
    if sampler:
        sampler.end()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, **out)
    sharding.barrier()
    launches = (_lib.launch_count() - launches0) // steps
    loop_ms = sharding.max_over_ranks(att.loop_ms / steps)
    e2e_ms = sharding.max_over_ranks(wall * 1e3 / steps)
    clocks = sampler.stop() if sampler else {}
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    line = {"metric": HITADV_METRIC, "value": world * B / (loop_ms * 1e-3), "unit": "cloud-iterations/s", "n_gpus": world,
            "steps": steps, "warmup": max(5, args.warmup), "ms_per_step": loop_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": name, "batch_per_gpu": B, "points": K, "attack_iters_per_s_per_batch": 1e3 / loop_ms,
                       "note": "value = device time of the iteration loop (CUDA events); e2e = whole attack() call: host data "
                               "in, one-off centre selection, iterations, adversarial clouds back to the host"},
            "clocks": clocks,
            "e2e": {"value": world * B / (e2e_ms * 1e-3), "unit": "cloud-iterations/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(data.numel() * 4 / steps), "d2h_bytes_per_step": int(B * K * 3 * 8 / steps)},
            "gpu_launches": int(launches)}
    if world == 1 and not args.no_cpu_baseline:
        try:  # the reference's torch program on THIS GPU (the second bar of BASELINE.md section 4)
            from oracle import hitadv_port as hp

            torch.manual_seed(0)
            n_ref = args.steps
            torch.cuda.synchronize()
            t0 = time.time()
            hp.attack(model, data.to(dev), target.to(dev), dict(HITADV_HP, kappa=30.0, binary_step=1, num_iter=n_ref))
            torch.cuda.synchronize()
            t_all = time.time() - t0
            t0 = time.time()
            hp.attack(model, data.to(dev), target.to(dev), dict(HITADV_HP, kappa=30.0, binary_step=1, num_iter=2 * n_ref))
            torch.cuda.synchronize()
            per_iter = (time.time() - t0 - t_all) / n_ref  # difference of two runs removes the one-off setup
            line["reference_torch_path_on_this_gpu"] = {"value": B / per_iter, "unit": "cloud-iterations/s",
                                                        "ms_per_step": per_iter * 1e3,
                                                        "what": "oracle/hitadv_port.py (the reference's tensor program) on cuda:0, batch %d" % B}
        except Exception as e:
            line["reference_torch_path_on_this_gpu"] = {"value": None, "what": f"failed: {e}"}
        try:
            r = hitadv_cpu(8, K, args.steps)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": "cloud-iterations/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# The caller of BASELINE config 1: the CW-kNN attack loop (CW/kNN.py) with ChamferkNNDist on 388 x 1024-point clouds
# against a random-init PointNet.  A "step" = one attack iteration over the batch (victim fwd/bwd -> Chamfer + kNN
# losses fwd/bwd -> Adam -> l_inf clip).  value = cloud-iterations per second.
# ------------------------------------------------------------------------------------------------------------
CWKNN_METRIC = "CW-kNN attack cloud-iterations/sec"
CWKNN_HP = dict(attack_lr=1e-3, kappa=15.0, budget=0.18)


def cwknn_inputs(B, K, seed):
    ori, _ = make_clouds(B, K, seed)
    rng = np.random.default_rng(seed + 1)
    return torch.from_numpy(ori), torch.from_numpy(rng.integers(0, 40, B))


def cwknn_port_run(B, K, iters, device):
    """The reference loop (oracle/cwknn_port.py + oracle/torch_port.py, bit-identical to the reference classes on CPU)
    -> (seconds, {"adv": adversarial clouds, "success": success count})."""
    from hitgeom import adv_utils, clip_utils
    from oracle import cwknn_port, torch_port
    from util_models import PointNetCls

    data, target = cwknn_inputs(B, K, 4321)
    model = PointNetCls(40, seed=0)
    torch.manual_seed(0)
    sync = torch.cuda.synchronize if device != "cpu" else (lambda: None)
    sync()
    t0 = time.time()
    adv, succ = cwknn_port.attack(model, data, target, adv_utils.LogitsAdvLoss(kappa=CWKNN_HP["kappa"]),
                                  torch_port.chamfer_knn_dist, clip_utils.ClipPointsLinf(budget=CWKNN_HP["budget"]),
                                  attack_lr=CWKNN_HP["attack_lr"], num_iter=iters, device=device)
    sync()
    return time.time() - t0, {"adv": adv, "success": np.float64(succ)}


def main_cwknn(args):
    from util_models import PointNetCls

    B, K = (args.clouds or 388), (args.points or 1024)
    name = f"C1 caller: CW-kNN attack loop (ChamferkNNDist, l_inf clip), batch {B} x {K} points, random-init PointNet victim"
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return
        torch.set_num_threads(os.cpu_count() or 1)
        Bc, it = 16, args.steps
        dt, out = cwknn_port_run(Bc, K, it, "cpu")
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, **out)
        cb = {"value": Bc * it / dt, "unit": "cloud-iterations/s", "cores": os.cpu_count(), "kind": "port",
              "sample": f"batch of {Bc} clouds x {K} points, {it} iterations"}
        line = {"impl": "reference", "metric": CWKNN_METRIC, "value": cb["value"], "unit": cb["unit"], "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / it * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": name},
                "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": cb["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return
    from hitgeom import _lib, sharding
    from hitgeom.adv_utils import LogitsAdvLoss
    from hitgeom.clip_utils import ClipPointsLinf
    from hitgeom.cw_knn import CWKNN
    from hitgeom.dist_utils import ChamferkNNDist

    rank, world, local = sharding.init()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    data, target = cwknn_inputs(B, K, 1234 + rank)
    model = PointNetCls(40, seed=0).to(dev)
    iters = args.steps
    n_graph = iters + CAPTURED_AFTER  # the timed graph-mode call replays `iters` iterations after its eager lead-in

    def run(n_iter, graph):
        att = CWKNN(model, LogitsAdvLoss(kappa=CWKNN_HP["kappa"]), ChamferkNNDist(), ClipPointsLinf(budget=CWKNN_HP["budget"]),
                    attack_lr=CWKNN_HP["attack_lr"], num_iter=n_iter, graph=graph)
        torch.manual_seed(0)
        torch.cuda.synchronize()
        t0 = time.time()
        adv, succ = att.attack(data, target)
        torch.cuda.synchronize()
        return att, time.time() - t0, {"adv": adv, "success": np.float64(succ)}

    run(max(8, args.warmup), True)
    run(max(8, args.warmup), False)
    sampler = ClockSampler(local) if rank == 0 else None
    sharding.barrier()
    if sampler:
        sampler.begin()
    att2, wall2, out = run(n_graph, True)
    if sampler:
        sampler.end()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, **out)
    sharding.barrier()
    launches0 = _lib.launch_count()
    att_e, _, _ = run(iters, False)
    launches = (_lib.launch_count() - launches0) // iters
    graph_ms = sharding.max_over_ranks(att2.replay_ms / max(att2.replays, 1))
    eager_ms = sharding.max_over_ranks(att_e.loop_ms / iters)
    e2e_ms = sharding.max_over_ranks(wall2 * 1e3 / n_graph)
    clocks = sampler.stop() if sampler else {}
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    line = {"metric": CWKNN_METRIC, "value": world * B / (graph_ms * 1e-3), "unit": "cloud-iterations/s", "n_gpus": world,
            "steps": int(att2.replays), "warmup": max(8, args.warmup), "ms_per_step": graph_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": name, "batch_per_gpu": B, "points": K, "eager_ms_per_step": eager_ms,
                       "note": "value = device time per iteration with the iteration replayed as one CUDA graph (CUDA events "
                               "around the replayed iterations of one attack() call); eager_ms_per_step = same loop launched kernel by kernel; e2e = whole "
                               "attack() call: host data in, iterations, adversarial clouds back to the host",
                       "l2": "working set (victim activations, 388 x 1024 x 1024 floats per layer) exceeds the 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": world * B / (e2e_ms * 1e-3), "unit": "cloud-iterations/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(data.numel() * 4 / n_graph), "d2h_bytes_per_step": int(B * K * 3 * 4 / n_graph)},
            "gpu_launches": int(launches),
            "gpu_launches_note": "hitgeom kernel launches per iteration, counted on the eager run (a graph replay re-runs the same kernels without passing the counter)"}
    if world == 1 and not args.no_cpu_baseline:
        try:  # the reference's torch program on THIS GPU
            n_ref = args.steps
            cwknn_port_run(B, K, 3, dev)
            per_iter = cwknn_port_run(B, K, n_ref, dev)[0] / n_ref
            line["reference_torch_path_on_this_gpu"] = {"value": B / per_iter, "unit": "cloud-iterations/s", "ms_per_step": per_iter * 1e3,
                                                        "what": "oracle/cwknn_port.py + torch_port.py (the reference's tensor program) on cuda:0, batch %d" % B}
        except Exception as e:
            line["reference_torch_path_on_this_gpu"] = {"value": None, "what": f"failed: {e}"}
        try:
            torch.set_num_threads(os.cpu_count() or 1)
            Bc, it = 16, args.steps
            dt, _ = cwknn_port_run(Bc, K, it, "cpu")
            line["cpu_baseline"] = {"value": Bc * it / dt, "unit": "cloud-iterations/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"batch of {Bc} clouds x {K} points, {it} iterations"}
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": "cloud-iterations/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.workload == "hitadv":
        main_hitadv(a)
    elif a.workload == "cwknn":
        main_cwknn(a)
    elif a.impl == "reference":
        main_reference(a)
    else:
        main_hitgeom(a)
