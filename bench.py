#!/usr/bin/env python
"""Benchmark of the cfm_b200 hot path on BASELINE.json's metric:
minibatch-OT couplings/sec (N=8192, d=784) [+ ODE samples/sec], 1..8 B200 of one node.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU path (oracle port) on host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's coupled batch to DIR/*.npy

One step = one full coupling `OTPlanSampler("sinkhorn", reg=0.05, normalize_cost=True).sample_plan`
(cost matrix + 100 log-domain Sinkhorn iterations, stopThr=0 + N pair draws + gather) on a
pair of synthetic Gaussian batches resident in HBM; weak scaling: every rank couples its own N=8192 shard
(per-shard coupling, the only collective is the NCCL all-gather of the sampled index pairs, issued on a side
stream).  Rank 0 prints ONE JSON line; besides the contract's keys it carries sub-records for the other BASELINE
configs (c1_coupling, c4, c5, ode, ode_c1, ode_strong), each with its parity gate.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N, D, REG, ITERS = 8192, 784, 0.05, 100
METRIC = "minibatch-OT couplings/sec (N=8192,d=784)"
WORKLOAD = ("C2: Sinkhorn minibatch coupling N=8192 d=784 fp32, 100 log-domain iterations "
            "(normalize_cost=True, reg=0.05, stopThr=0): cost matrix + solve + 8192 pair draws + gather")
ODE_B, ODE_DIM, ODE_W = 10000, 784, 256
REF_BUDGET_S = 150.0  # wall budget of the timed steps of `--impl reference` (each step is one FULL coupling)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md's clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(index)], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------ CPU reference arm
class CpuReference:
    """The reference's CPU path for one C2 coupling, restated (oracle/coupling.py + oracle/ot; POT itself is not
    installable here): torch.cdist**2 / max -> POT's KERNEL-SPACE sinkhorn_knopp with POT's dtype pattern (fp32 K,
    float64 Kp and vectors; this is what OTPlanSampler('sinkhorn') calls and it is finite in this normalised
    regime) for exactly 100 iterations -> u K v plan -> np.random.choice over the flattened plan -> gather.
    Every part is executed in full; nothing is extrapolated."""

    def __init__(self, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.x0, self.x1 = torch.randn(N, D, generator=g), torch.randn(N, D, generator=g)

    def coupling(self):
        from oracle import coupling as oc
        t = {}
        t0 = time.perf_counter()
        Mn = oc.cost_matrix(self.x0, self.x1, normalize_cost=True).detach().cpu().numpy()
        t["cost"] = time.perf_counter() - t0
        a = b = np.ones(N) / N
        t0 = time.perf_counter()
        K = np.exp(Mn / (-REG))                 # fp32
        Kp = (1 / a).reshape(-1, 1) * K         # float64 (POT dtype pattern)
        u = np.ones(N, dtype=Mn.dtype) / N
        t["setup"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        for _ in range(ITERS):
            v = b / np.dot(K.T, u)
            u = 1.0 / np.dot(Kp, v)
        t["iters"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        P = u.reshape((-1, 1)) * K * v.reshape((1, -1))
        i, j = oc.draw_pairs(P, N)
        _ = self.x0[i], self.x1[j]
        t["draw"] = time.perf_counter() - t0
        return sum(t.values()), t


def run_reference_arm(args, rank):
    """`bench.py --impl reference`: every step is ONE COMPLETE coupling of the reference's CPU path (kind "port":
    the oracle restatement, kernel-space Sinkhorn-Knopp like the reference) on all host cores.  A coupling takes tens
    of seconds here, so the number of timed steps is bounded by a wall budget (at least one, at most --steps) and
    reported as `steps`; `steps_requested` keeps the driver's K."""
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    ref = CpuReference(0)
    np.dot(np.ones((512, 512), np.float32), np.ones(512, np.float32))  # BLAS thread pool spin-up (the only warm-up)
    times, parts = [], None
    t_begin = time.perf_counter()
    while len(times) < max(1, args.steps):
        dt, parts = ref.coupling()
        times.append(dt)
        if time.perf_counter() - t_begin + dt > REF_BUDGET_S:
            break
    wall = time.perf_counter() - t_begin
    value = len(times) / sum(times)
    cores = os.cpu_count() or 1
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "couplings/s",
        "n_gpus": args.gpus, "steps": len(times), "steps_requested": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "solver": "kernel-space Sinkhorn-Knopp (POT sinkhorn_knopp restated), 100 iterations",
                   "note": "CPU path, one coupling stream regardless of --gpus; every step is a complete coupling; the "
                           "warm-up is the BLAS thread-pool spin-up only (a warm-up coupling would cost a whole step); "
                           f"timed wall {wall:.1f} s for {len(times)} step(s), budget {REF_BUDGET_S:.0f} s"},
        "cpu_baseline": {"value": value, "unit": "couplings/s", "cores": cores, "kind": "port",
                         "sample": f"{len(times)} complete N=8192,d=784 coupling(s): cdist**2/max, exp(-M/reg), 100 Knopp "
                                   "iterations (fp32 K, float64 Kp/u/v), plan, np.random.choice, gather; "
                                   f"parts(s) of the last one={ {k: round(v, 3) for k, v in parts.items()} }"},
        "e2e": {"value": value, "unit": "couplings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "step_ms": {"median": float(np.median(times) * 1e3), "min": float(min(times) * 1e3), "max": float(max(times) * 1e3)},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------ helpers (GPU arm)
def eight_gaussians(n, gen):
    """utils.sample_8gaussians restated (torchcfm/utils.py:11-41): radius-5 octagon, per-axis std 0.1**0.25."""
    ang = torch.arange(8) * (2 * np.pi / 8)
    centers = 5.0 * torch.stack([torch.cos(ang), torch.sin(ang)], 1)
    k = torch.randint(0, 8, (n,), generator=gen)
    return (centers[k] + (0.1 ** 0.25) * torch.randn(n, 2, generator=gen)).float()


def two_moons(n, gen):
    """utils.sample_moons restated (torchcfm/utils.py:35-37): generate_moons(n, noise=0.2) * 3 - 1."""
    n_out = n // 2
    to, ti = torch.linspace(0, np.pi, n_out), torch.linspace(0, np.pi, n - n_out)
    x = torch.cat([torch.stack([torch.cos(to), torch.sin(to)], 1),
                   torch.stack([1 - torch.cos(ti), 1 - torch.sin(ti) - 0.5], 1)], 0)
    x = x + 0.2 * torch.randn(n, 2, generator=gen)
    return (x[torch.randperm(n, generator=gen)] * 3 - 1).float()


def timed_ms(fn, reps, dev, warm=2):
    """Mean device time of fn() over `reps` back-to-back calls (CUDA events on the current stream)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


# ------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cfm_b200", choices=["cfm_b200", "reference"])
    ap.add_argument("--no-ode", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the c1/c4/c5 sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0's sample_plan pair "
                         "x0[i], x1[j], float32) as DIR/<name>.npy: the same arguments give the same inputs and draws, "
                         "so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "cfm_b200":
        ap.error("--dump-outputs writes the outputs of the cfm_b200 path")
    args.warmup = max(args.warmup, 3) if args.impl == "cfm_b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference_arm(args, rank)

    import torch.distributed as dist

    import cfm_b200
    from cfm_b200 import _ffi
    from cfm_b200 import dist as cdist
    from oracle import coupling as oc
    from oracle import vector_field as vf

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _ffi.require_device()  # raises if the library / an sm_100 device is missing: no fallback
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = _ffi.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # synthetic inputs: generated on the CPU (identical bits for the CPU baseline), distinct per rank
    g = torch.Generator().manual_seed(rank)
    x0_h = torch.randn(N, D, generator=g).pin_memory()
    x1_h = torch.randn(N, D, generator=g).pin_memory()
    x0, x1 = x0_h.to(dev), x1_h.to(dev)
    sampler = cfm_b200.OTPlanSampler("sinkhorn", reg=REG, normalize_cost=True, num_iter_max=ITERS,
                                     stop_thr=0.0, warn=False)
    np.random.seed(1234 + rank)

    pending = []

    def step():
        if world > 1:
            a, b, h = cdist.sharded_sample_plan(sampler, x0, x1, async_gather=True)
            pending.append(h)  # the index all-gather overlaps the next coupling; picked up below
            if len(pending) > 1:
                pending.pop(0).wait()
            return a, b
        return sampler.sample_plan(x0, x1)

    # nvidia-smi is started BEFORE the warm-up (its start-up stalls the GPU for a few ms) and keeps
    # sampling through the timed region
    clocks = ClockSampler(local_rank) if (rank == 0 and not os.environ.get("CFM_BENCH_NOCLK")) else None
    if clocks is not None:
        time.sleep(0.7)  # let nvidia-smi finish initialising NVML before any timed work
    out = None
    for _ in range(args.warmup):
        out = step()  # results stay alive for one step, as in the timed loop: the allocator's pools reach steady state
    barrier()

    # ---- timed region: K steps, device events, barrier + synchronize both sides ----
    sampler.stage_events = []
    launches0 = L.cfm_launch_count()
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    host_ms = []
    gc.collect()
    gc.disable()  # no collector pause inside the timed region (it is re-enabled right after)
    barrier()
    marks[0].record()
    for k in range(args.steps):
        th = time.perf_counter()
        out = step()
        marks[k + 1].record()
        host_ms.append((time.perf_counter() - th) * 1e3)
    while pending:
        pending.pop(0).wait()
    barrier()
    gc.enable()
    elapsed_ms = marks[0].elapsed_time(marks[-1])
    per_step = [marks[k].elapsed_time(marks[k + 1]) for k in range(args.steps)]
    launches = L.cfm_launch_count() - launches0
    clk = clocks.stop() if clocks else None
    stage_ms = {}
    for name, a, b in sampler.stage_events:
        stage_ms.setdefault(name, []).append(a.elapsed_time(b))
    sampler.stage_events = None
    elapsed_ms = max_over_ranks(elapsed_ms)
    value = world * args.steps / (elapsed_ms * 1e-3)
    assert out[0].shape == (N, D) and out[0].is_cuda
    if args.dump_outputs and rank == 0:  # 2 x 8192 x 784 float32 = 51 MB
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in zip(("x0_coupled", "x1_coupled"), out):
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), t.float().cpu().numpy())

    # ---- parity gate reported with the number: marginals of the implied plan (float64, device)
    cp = sampler._couple(x0, x1, dev)
    Mn = (cp.M[:, :N] / cp.cost_max).double()
    P = (-(Mn / REG) + cp.log_u[:, None] + cp.log_v[None, :]).exp()
    parity = {"row_marginal_max_rel_err": float((P.sum(1) * N - 1).abs().max().item()),
              "col_marginal_max_rel_err": float((P.sum(0) * N - 1).abs().max().item()),
              "iterations": int(cp.status[1].item())}
    del P, Mn, cp

    # ---- e2e: public API with HOST (pinned) inputs; H2D + D2H of every step inside the timed region ----
    # (1) blocking call: sampler.sample_plan(host, host) -> host, one batch at a time
    for _ in range(2):
        sampler.sample_plan(x0_h, x1_h)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        a_h, b_h = sampler.sample_plan(x0_h, x1_h)
    torch.cuda.synchronize(dev)
    single_s = time.perf_counter() - t0
    # (2) the streaming form of the same call (cfm_b200.CouplingStream): every step still uploads its
    # inputs and downloads its coupled batch, but batch k+1's upload and batch k-1's download overlap
    # batch k's solve on separate streams.  This is the headline e2e number.
    from cfm_b200 import CouplingStream
    pipe = CouplingStream(sampler, dev, depth=2)
    warm = 6
    n_out = -warm
    t0 = None
    barrier()
    for a_h, b_h in pipe.map((x0_h, x1_h) for _ in range(warm + args.steps)):
        n_out += 1
        if n_out == 0:
            t0 = time.perf_counter()
    e2e_s = time.perf_counter() - t0
    torch.cuda.synchronize(dev)
    assert n_out == args.steps
    e2e_s, single_s = max_over_ranks(e2e_s), max_over_ranks(single_s)
    e2e = {"value": world * args.steps / e2e_s, "unit": "couplings/s",
           "h2d_bytes_per_step": int(2 * N * D * 4 + N * 8), "d2h_bytes_per_step": int(2 * N * D * 4),
           "api": "CouplingStream(sampler).map(host batches), depth 2; K consecutive steady-state results timed "
                  "after 6 untimed ones of the same stream",
           "blocking_call_value": world * args.steps / single_s}
    assert a_h.device.type == "cpu" and a_h.shape == (N, D)

    # ---- roofline of the dominant kernel (the persistent Sinkhorn sweep kernel) + the tensor-core kernels ----
    hbm_peak, tc_peak, which = peaks()
    solve_ms = float(np.mean(stage_ms["solve"]))
    cost_ms = float(np.mean(stage_ms["cost"]))
    one_pass = ITERS * N * N * 4  # the fused sweep reads M once per iteration (row AND column update per pass)
    achieved = one_pass / (solve_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("sinkhorn_kernel_dram_bytes_per_launch")
    kernels = [{"kernel": "gemm_h3_kernel<128, SqDistH3Epilogue> + 2 prep_rows_h3 (stage 'cost')", "bound": "tensor",
                "ms": cost_ms, "algorithmic_tflops": 2.0 * N * N * D / (cost_ms * 1e-3) / 1e12,
                "issued_tflops_f16": 3 * 2.0 * N * N * D / (cost_ms * 1e-3) / 1e12, "peak_tflops_f16": tc_peak,
                "frac_issued": 3 * 2.0 * N * N * D / (cost_ms * 1e-3) / 1e12 / tc_peak,
                "note": "fp16x3 scheme: three kind::f16 MMAs per product for fp32-grade accuracy; the stage time "
                        "includes the two row pre-passes (norms, scales, operand split)"}]
    roofline = {"bound": "hbm", "kernel": "sinkhorn_v2_kernel<512,4,2> (100 fused sweeps, one cooperative launch)",
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "frac_one_pass": achieved / hbm_peak,
                "frac_dram": (traffic / (solve_ms * 1e-3) / 1e9 / hbm_peak) if traffic else None,
                "traffic": traffic, "peak_source": which,
                "algorithmic_bytes": one_pass,
                "survey_8d": {"bytes": 2 * one_pass, "gbs": 2 * achieved,
                              "note": "SURVEY 8(d) counts two passes over M per iteration; the fused sweep makes one, "
                                      "so this figure is a labelled aside, not a fraction of peak"},
                "note": "frac = one-pass algorithmic bytes (iters*N^2*4) / solve time / measured HBM peak; frac_dram "
                        "= ncu DRAM bytes of the same kernel (profiles/roofline_traffic.json) / solve time / peak: "
                        "part of M stays L2-resident between sweeps, so DRAM traffic is below the one-pass bytes",
                "stage_ms": {k: float(np.mean(v)) for k, v in stage_ms.items()},
                "kernels": kernels}

    line = {
        "metric": METRIC, "value": value, "unit": "couplings/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "per_gpu_batch": N, "dim": D, "parallelism": f"shard{world}",
                   "l2": "inputs larger than L2: the cost matrix streamed every iteration is 268 MB"},
        "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
        "parity": parity,
        "step_ms": {"median": float(np.median(per_step)), "min": float(min(per_step)), "max": float(max(per_step)),
                    "host_enqueue_ms_max": float(max(host_ms)), "host_enqueue_ms_median": float(np.median(host_ms)),
                    "note": "per-step device time of rank 0 (events between steps); host_enqueue_ms = wall time the host "
                            "spent inside each (asynchronous) sample_plan call"},
    }

    # ---- the other BASELINE configs, each with its parity gate (rank-local work; max over ranks reported) ----
    if not args.no_extra:
        # C1: 8gaussians -> 2moons, exact OT, batch 256 (examples/2D_tutorials)
        gen = torch.Generator().manual_seed(10 + rank)
        a8, m2 = eight_gaussians(256, gen), two_moons(256, gen)
        a8d, m2d = a8.to(dev), m2.to(dev)
        ex = cfm_b200.OTPlanSampler("exact")
        pi = ex.get_map(a8d, m2d)
        sig_ok = bool(np.array_equal(pi.argmax(1), oc.assignment(oc.cost_matrix(a8, m2))))
        np.random.seed(77)
        c1_ms = timed_ms(lambda: ex.sample_plan(a8d, m2d), 50, dev, warm=5)
        t0 = time.perf_counter()
        for _ in range(20):
            np.random.seed(77)
            oc.sample_plan(a8, m2, "exact")
        c1_cpu_ms = (time.perf_counter() - t0) / 20 * 1e3
        line["c1_coupling"] = {"config": "C1: 8gaussians->2moons exact OT coupling, batch 256, d=2 (cost + exact assignment "
                                         "+ 256 pair draws + gather, status word read every call)",
                               "ms_per_coupling": max_over_ranks(c1_ms), "couplings_per_s": world * 1e3 / max_over_ranks(c1_ms),
                               "sigma_bit_exact_vs_scipy": sig_ok, "dijkstra_steps": ex.last_info.get("dijkstra_steps"),
                               "cpu_reference_port_ms": c1_cpu_ms if rank == 0 else None}

        # C4: SB-CFM entropic OT eps = 2 sigma^2 = 0.1, N = 16384 d = 512 in 4 shards of 4096 (per-shard coupling)
        fm = cfm_b200.SchrodingerBridgeConditionalFlowMatcher(sigma=0.05 ** 0.5, ot_method="sinkhorn")
        sb = fm.ot_sampler
        sb.num_iter_max, sb.stop_thr, sb.warn = 100, 0.0, False
        g4 = torch.Generator().manual_seed(40 + rank)
        y0, y1 = torch.randn(4096, 512, generator=g4).to(dev), torch.randn(4096, 512, generator=g4).to(dev)
        np.random.seed(4)
        c4_ms = timed_ms(lambda: sb.sample_plan(y0, y1), 5, dev, warm=2)
        cp4 = sb._couple(y0, y1, dev)
        i4, j4 = sb._draw(cp4, 4096)
        Mr = -(cp4.M[:, :4096] / np.float32(sb.reg)).double()
        P4 = (Mr + cp4.log_u[:, None] + cp4.log_v[None, :]).exp()
        st4 = cp4.status.cpu().tolist()
        line["c4"] = {"config": "C4: SB-CFM entropic coupling eps=0.1 (un-normalised cost, |M/eps| ~ 1e4: float64-potential "
                                "mode), shards of 4096 x 4096, d=512, 100 iterations, one shard per GPU "
                                f"({world} shard(s) in this run; BASELINE: 4)",
                      "ms_per_shard_coupling": max_over_ranks(c4_ms), "shard_couplings_per_s": world * 1e3 / max_over_ranks(c4_ms),
                      "arithmetic": {0: "fp32", 1: "fp64", 2: "fp64-mixed"}.get(st4[2], st4[2]),
                      "solver": {0: "generic sweep", 1: "seeded fp32 screening (thresholds from the previous iteration's "
                                 "log-sum-exps; only the plan's support takes the float64 path)"}.get(st4[3], st4[3]),
                      "row_marginal_max_rel_err": float((P4.sum(1) * 4096 - 1).abs().max().item()),
                      "draw_flags": st4[0] & 3,
                      "note": "row marginals are exact by construction after the final row update; the column marginals of "
                              "this un-converged regime are far from uniform after 100 iterations for ANY log-domain solver "
                              "(SURVEY finding 11-ii); the reference's own kernel-space path underflows here and silently "
                              "returns the uniform plan"}
        del P4, Mr, cp4

        # C5: Sinkhorn sweep N in {1k, 4k, 16k, 64k} d = 128 over 8 shards -> per-shard sizes 128 ... 8192
        c5 = []
        s5 = cfm_b200.OTPlanSampler("sinkhorn", reg=REG, normalize_cost=True, num_iter_max=ITERS, stop_thr=0.0, warn=False)
        for ns in (128, 512, 2048, 8192):
            g5 = torch.Generator().manual_seed(50 + rank + ns)
            z0, z1 = torch.randn(ns, 128, generator=g5).to(dev), torch.randn(ns, 128, generator=g5).to(dev)
            np.random.seed(5)
            ms = timed_ms(lambda: s5.sample_plan(z0, z1), 10 if ns < 8192 else 5, dev, warm=2)
            cp5 = s5._couple(z0, z1, dev)
            P5 = (-((cp5.M[:, :ns] / cp5.cost_max).double() / REG) + cp5.log_u[:, None] + cp5.log_v[None, :]).exp()
            c5.append({"n_global_at_8_shards": 8 * ns, "n_per_shard": ns, "ms_per_shard_coupling": max_over_ranks(ms),
                       "pairs_per_s": world * ns * 1e3 / max_over_ranks(ms),
                       "col_marginal_max_rel_err": float((P5.sum(0) * ns - 1).abs().max().item())})
            del P5, cp5
        line["c5"] = {"config": f"C5: Sinkhorn sweep d=128, reg=0.05 normalised, 100 iterations, per-shard sizes of the "
                                f"8-way sharded N in {{1k,4k,16k,64k}}; {world} shard(s) in this run (BASELINE: 8)",
                      "sweep": c5}

    # ---- second half of the metric: ODE samples/sec (BASELINE config 3) ----
    if not args.no_ode:
        torch.manual_seed(0)
        mlp = cfm_b200.MLP(dim=ODE_DIM, w=ODE_W, time_varying=True).to(dev)
        node = cfm_b200.NeuralODE(cfm_b200.torch_wrapper(mlp), solver="dopri5", atol=1e-4, rtol=1e-4)
        xo = torch.randn(ODE_B, ODE_DIM, generator=torch.Generator().manual_seed(100 + rank)).to(dev)
        span = torch.linspace(0, 1, 2)
        for _ in range(3):
            node.trajectory(xo, span)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            node.trajectory(xo, span)
        e1.record()
        barrier()
        ode_s = max_over_ranks(e0.elapsed_time(e1)) * 1e-3 / reps
        nfe = node.stats["nfe"]
        flops = 2.0 * ODE_B * (785 * 256 + 256 * 256 + 256 * 256 + 256 * 784) * nfe
        # the forward alone (one fused launch + the fp32 -> fp16x3 split of its input), replayed from a CUDA graph
        # so that the host's per-call Python work does not sit between the launches
        yb = torch.empty_like(xo)
        t_dev = torch.full((1,), 0.5, dtype=torch.float32, device=dev)
        mlp.vector_field(t_dev, xo, out=yb)
        torch.cuda.synchronize(dev)
        gfwd = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gfwd):
            mlp.vector_field(t_dev, xo, out=yb)
        fwd_ms = timed_ms(gfwd.replay, 50, dev, warm=5)
        fwd_flops = 2.0 * ODE_B * (785 * 256 + 256 * 256 + 256 * 256 + 256 * 784)
        line["ode"] = {"metric": "ODE samples/sec (MLP 785-256-256-256-784 SELU, dopri5 atol=rtol=1e-4, B=10000/GPU)",
                       "value": world * ODE_B / ode_s, "unit": "samples/s", "nfe": nfe,
                       "accepted": node.stats["accepted"], "rejected": node.stats["rejected"],
                       "ms_per_trajectory": ode_s * 1e3, "mlp_tflops_algorithmic": flops / ode_s / 1e12,
                       "mlp_rows_per_s_per_nfe": world * ODE_B * nfe / ode_s,
                       "mlp_launches_per_nfe": 1 if mlp.w == 256 else 4,
                       "mlp_forward_ms": fwd_ms}
        roofline["kernels"].append({"kernel": "mlp_fused_h3_kernel (whole 4-layer forward, one launch) + input split",
                                    "bound": "tensor", "ms": fwd_ms,
                                    "algorithmic_tflops": fwd_flops / (fwd_ms * 1e-3) / 1e12,
                                    "issued_tflops_f16": 3 * fwd_flops / (fwd_ms * 1e-3) / 1e12, "peak_tflops_f16": tc_peak,
                                    "frac_issued": 3 * fwd_flops / (fwd_ms * 1e-3) / 1e12 / tc_peak,
                                    "note": "79 row slabs of 128 on 148 SMs (B = 10000): at most 53% of the tensor pipes "
                                            "can be busy in this one-slab-per-CTA design"})
        if rank == 0:
            # comparator on the same GPU: stock PyTorch eager (cuBLAS sgemm, TF32 off) through the
            # oracle's torchdyn-style driver
            torch.backends.cuda.matmul.allow_tf32 = False
            ref_m = vf.make_mlp(ODE_DIM, w=ODE_W, time_varying=True).to(dev)
            ref_m.load_state_dict(mlp.state_dict())
            f = lambda t, z: vf.wrapped_forward(ref_m, t, z)  # noqa: E731
            for _ in range(2):
                vf.dopri5_trajectory(f, xo, span.to(dev))
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for _ in range(3):
                vf.dopri5_trajectory(f, xo, span.to(dev))
            torch.cuda.synchronize(dev)
            line["ode"]["torch_eager_same_gpu_samples_per_s"] = ODE_B / ((time.perf_counter() - t0) / 3)
        barrier()

        # ---- strong scaling of C3 with row sharding (SURVEY 8e): B = 10000 split over the ranks ----
        if world > 1:
            xg = torch.randn(ODE_B, ODE_DIM, generator=torch.Generator().manual_seed(100)).to(dev)  # same on all ranks
            res = {}
            for mode, lock in (("lockstep", True), ("independent", False)):
                for _ in range(2):
                    cdist.sharded_trajectory(node, xg, span, gather=False, lockstep=lock)
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    cdist.sharded_trajectory(node, xg, span, gather=False, lockstep=lock)
                e1.record()
                barrier()
                s_ = max_over_ranks(e0.elapsed_time(e1)) * 1e-3 / 5
                res[mode] = {"samples_per_s": ODE_B / s_, "ms_per_trajectory": s_ * 1e3, "nfe": node.stats["nfe"],
                             "accepted": node.stats["accepted"], "rejected": node.stats["rejected"]}
            line["ode_strong"] = dict(res, config=f"C3 strong scaling: B = {ODE_B} rows split over {world} ranks "
                                                  "(weights replicated); lockstep = one float64 all-reduce per step attempt, "
                                                  "step sequence of the single-process run; independent = per-shard controllers")

        # ---- BASELINE config 1 sampling: the 2-D tutorial model, launch-bound regime (SURVEY 8 f-2) ----
        torch.manual_seed(0)
        small = cfm_b200.MLP(dim=2, w=64, time_varying=True).to(dev)
        nsm = cfm_b200.NeuralODE(cfm_b200.torch_wrapper(small), solver="dopri5", atol=1e-4, rtol=1e-4)
        xs = torch.randn(1024, 2, generator=torch.Generator().manual_seed(7)).to(dev)
        span100 = torch.linspace(0, 1, 100)
        for _ in range(3):
            nsm.trajectory(xs, span100)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(20):
            nsm.trajectory(xs, span100)
        torch.cuda.synchronize(dev)
        c1_s = (time.perf_counter() - t0) / 20
        line["ode_c1"] = {"metric": "ODE samples/sec (MLP 3-64-64-64-2 SELU, dopri5 1e-4, B=1024, 100 t_span points)",
                          "value": world * 1024 / c1_s, "unit": "samples/s", "ms_per_trajectory": c1_s * 1e3,
                          "nfe": nsm.stats["nfe"], "launches_per_trajectory": 1 if nsm.stats.get("fused") else None}
        if rank == 0:
            ref_s = vf.make_mlp(2, w=64, time_varying=True).to(dev)
            ref_s.load_state_dict(small.state_dict())
            fs = lambda t, z: vf.wrapped_forward(ref_s, t, z)  # noqa: E731
            with torch.no_grad():
                vf.dopri5_trajectory(fs, xs, span100.to(dev))
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                vf.dopri5_trajectory(fs, xs, span100.to(dev))
                torch.cuda.synchronize(dev)
            line["ode_c1"]["torch_eager_same_gpu_samples_per_s"] = 1024 / (time.perf_counter() - t0)

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only): ONE complete coupling, nothing extrapolated ----
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        np.dot(np.ones((512, 512), np.float32), np.ones(512, np.float32))
        dt, parts = CpuReference(0).coupling()
        line["cpu_baseline"] = {
            "value": 1.0 / dt, "unit": "couplings/s", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": "one COMPLETE N=8192,d=784 coupling of the reference CPU path restated (torch.cdist**2/max, POT "
                      "kernel-space sinkhorn_knopp in NumPy with POT's dtype pattern, 100 iterations, np.random.choice, "
                      f"gather), nothing extrapolated; parts(s)={ {k: round(x, 3) for k, x in parts.items()} }"}
    elif rank == 0:
        line["cpu_baseline"] = None

    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
