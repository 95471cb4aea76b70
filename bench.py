#!/usr/bin/env python
"""bench.py -- graph-trajectory solver steps/sec (fwd+bwd) of the fused sm_100a hot path.

One bench "step" = one forward + exact-adjoint backward solve of a batch of B graph trajectories
(S Tsit5 steps each) per GPU.  value = N_gpus * B * S / seconds_per_bench_step  (whole-job aggregate).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference]

N > 1 is launched by torchrun (one rank per GPU, NCCL); the batch of trajectories is sharded over the
ranks (weak scaling: B graphs per GPU) and the flat parameter-gradient buffer is all-reduced every step.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# name -> shape.  The C5 sweep points are BASELINE.json configs[4]; sir / england / twitter are configs[1..3].
WORKLOADS = {
    "sir": dict(n=100, h=32, e=3, L=3, T=120, t1=1.0, dt0=0.1, B=50, float_ts=True),
    "england": dict(n=129, h=64, e=8, L=3, T=4, t1=3.0, dt0=0.1, B=1),
    "twitter": dict(n=1000, h=64, e=16, L=3, T=9, t1=8.0, dt0=0.1, B=1),
    # graphs per GPU are chosen so that (row blocks of 128) x B is just under a multiple of the 148 SMs
    "sweep_n1024_h64": dict(n=1024, h=64, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=18),
    "sweep_n1024_h256": dict(n=1024, h=256, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=18),
    "sweep_n1024_h128_e8": dict(n=1024, h=128, e=8, L=3, T=9, t1=8.0, dt0=0.1, B=18),
    "sweep_n4096_h64": dict(n=4096, h=64, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=9),
    "sweep_n16384_h64": dict(n=16384, h=64, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=1),
    "sweep_n2048_h64": dict(n=2048, h=64, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=9),
    "sweep_n2048_h128": dict(n=2048, h=128, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=9),
    "sweep_n4096_h128": dict(n=4096, h=128, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=9),
    "sweep_n4096_h128_b4": dict(n=4096, h=128, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=4),
    "sweep_n4096_h256": dict(n=4096, h=256, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=4),
    "sweep_n8192_h128": dict(n=8192, h=128, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=2),
    "sweep_n16384_h128": dict(n=16384, h=128, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=1),
    "sweep_n16384_h256": dict(n=16384, h=256, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=1),
}
DEFAULT_WORKLOAD = "sweep_n2048_h128"
METRIC = "graph-trajectory solver steps/sec (fwd+bwd)"
UNIT = "solver steps/s"


def measured_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel (mean of one forward and one
    adjoint launch), from the committed `ncu --set full` captures of this workload (profiles/r02_traffic.json);
    None if no capture exists."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(path):
        ent = json.load(open(path)).get(workload)
        return ent["mean_bytes_per_launch"] if isinstance(ent, dict) else ent
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=float(d["hbm_gbs"]), bf16=float(d["bf16_tflops_sustained"]), src="measured")
    return dict(hbm=6650.0, bf16=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, threading.Event(), []

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def synth_adjacency(n, T, seed, device):
    """Device-side synthetic dynamic weighted digraph [T,n,n] (SURVEY 8(d)): Bernoulli(min(1,16/n)) mask with
    10% of entries redrawn per knot, LogNormal(0,1) weights, unit self-loops, row-normalised."""
    g = torch.Generator(device=device).manual_seed(seed)
    p = min(1.0, 16.0 / n)
    mask = torch.rand((n, n), generator=g, device=device) < p
    w = torch.exp(torch.randn((n, n), generator=g, device=device))
    out = torch.empty((T, n, n), device=device)
    eye = torch.eye(n, device=device, dtype=torch.bool)
    for k in range(T):
        if k > 0:
            redraw = torch.rand((n, n), generator=g, device=device) < 0.10
            mask = torch.where(redraw, torch.rand((n, n), generator=g, device=device) < p, mask)
            w = torch.where(redraw, torch.exp(torch.randn((n, n), generator=g, device=device)), w)
        a = torch.where(mask, w, torch.zeros_like(w))
        a = torch.where(eye, torch.ones_like(a), a)
        out[k] = a / a.sum(dim=1, keepdim=True)
    return out


def make_inputs(wl, seed, device, host_copy, coeff_budget=None):
    """Inputs of one rank.  Reference layout: ts [T], coeffs_adj (d,c,b,a) each [B,T-1,n,n,2], x_coeffs, y0, cotangent -- plus the
    graph snapshots A_k [B,T,n,n] they were built from.  The reference-layout arrays are 32 n^2 (T-1) bytes per graph; past
    COEFF_BUDGET bytes (n = 16384: 69 GB) only the snapshots are kept and the control path is built on the device
    (pegncde_build_adj, bit-identical planes)."""
    import perm_equiv_graph_neural_cdes_b200 as P

    n, h, e, T, B = wl["n"], wl["h"], wl["e"], wl["T"], wl["B"]
    ts = torch.linspace(0.0, wl["t1"], T, device=device) if wl.get("float_ts") else torch.arange(T, device=device, dtype=torch.float32) * (wl["t1"] / (T - 1))
    coeff_bytes = 4 * B * (T - 1) * n * n * 2 * 4
    with_coeffs = coeff_bytes <= (COEFF_BUDGET if coeff_budget is None else coeff_budget)
    cadj = [torch.empty((B, T - 1, n, n, 2), device=device) for _ in range(4)] if with_coeffs else None
    snaps_dev = None if with_coeffs else torch.empty((B, T, n, n), device=device)
    snaps = torch.empty((B, T, n, n), dtype=torch.float32).pin_memory() if host_copy else None
    for b in range(B):
        A = synth_adjacency(n, T, seed * 1000 + b, device)
        if snaps is not None:
            snaps[b].copy_(A)
        if with_coeffs:
            X = torch.stack([ts[:, None, None].expand(T, n, n), A], dim=-1)
            for dst, src in zip(cadj, P.backward_hermite_coefficients(ts, X)):
                dst[b].copy_(src)
            del X
        else:
            snaps_dev[b].copy_(A)
        del A
    g = torch.Generator(device=device).manual_seed(seed + 77)
    xco, x_t = None, None
    if e > 0:
        x_t = 0.3 * torch.randn((B, T, n, e), generator=g, device=device)
        X = torch.stack([ts[None, :, None, None].expand(B, T, n, e), x_t], dim=-1)
        xco = [torch.stack([P.backward_hermite_coefficients(ts, X[b])[i] for b in range(B)]) for i in range(4)]
    y0 = torch.randn((B, n, h), generator=g, device=device)
    gy = torch.randn((B, n, h), generator=g, device=device)
    host = None
    if host_copy:
        pin = lambda t: t.cpu().pin_memory()
        host = dict(ts=pin(ts), cadj=[pin(c) for c in cadj] if with_coeffs else None, xco=None if xco is None else [pin(c) for c in xco], y0=pin(y0),
                    snaps=snaps, x_t=None if e == 0 else pin(x_t))
    return ts, cadj, xco, y0, gy, host, snaps_dev, x_t


COEFF_BUDGET = 40e9
DUMP_BUDGET = 63_000_000   # bytes of array data written by --dump-outputs (the .npy headers keep the total under 64 MB)


def dump_outputs(out_dir, arrays, budget=DUMP_BUDGET):
    """Writes every array as `out_dir/<name>.npy` in float32.  If all of them together exceed `budget` bytes, each array is cut to
    the same fraction of its elements, taken flat at positions drawn with a fixed seed (sorted), so that two builds of the project
    run with the same arguments write values from the same positions and can be compared output for output."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    total = 4 * sum(a.numel() for a in arrays.values())
    for name, a in arrays.items():
        a = a.detach().float()
        if total > budget:
            keep = max(1, a.numel() * budget // total)
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            a = a.reshape(-1)[idx.to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def tensor_peaks(dev):
    """Dense GEMM throughput of cuBLAS on this GPU, measured live (8192^3, best of 5 after warm-up): tf32 (fp32 inputs with
    allow_tf32) and fp16 / bf16 -- the denominators of the executed-tensor-work fractions reported beside the HBM roofline."""
    out = {}
    N = 8192
    for name, dt, tf in (("tf32", torch.float32, True), ("fp16", torch.float16, False), ("bf16", torch.bfloat16, False)):
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = tf
        a = torch.randn((N, N), device=dev, dtype=dt)
        b = torch.randn((N, N), device=dev, dtype=dt)
        c = torch.empty((N, N), device=dev, dtype=dt)
        for _ in range(2):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a, b, out=c); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        out[name] = 2.0 * N ** 3 / (best * 1e-3) / 1e12
        torch.backends.cuda.matmul.allow_tf32 = prev
        del a, b, c
    torch.cuda.empty_cache()
    return out


class Dist:
    """Rank bookkeeping of one bench process (torchrun env: RANK / LOCAL_RANK / WORLD_SIZE)."""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            torch.distributed.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_ms(self, ms):
        t = torch.tensor([ms], device=self.dev)
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())


def operand_flags(args):
    from perm_equiv_graph_neural_cdes_b200 import _lib

    flags = 0 if args.no_tensor_cores else _lib.PEG_FLAG_TENSOR_CORES
    if args.tf32_fast:
        flags |= _lib.PEG_FLAG_TF32_FAST
    if args.operands == "tf32x3":
        flags |= _lib.PEG_FLAG_TF32X3
    elif args.operands == "bf16x2":
        flags |= _lib.PEG_FLAG_BF16X2
    return flags


def measure_fixed(D, wl_name, wl, args, steps, warmup, with_e2e, tpeaks, e2e_steps, coeff_budget=None, dump_dir=None):
    """One fixed-step workload on this rank's GPU: device-resident value (CUDA-graph replay), the roofline of the contraction
    launches, and (optionally) the end-to-end legs from pinned host buffers.  Returns a dict (rank-local; times are max over ranks).
    With `dump_dir`, rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    import perm_equiv_graph_neural_cdes_b200 as P
    from perm_equiv_graph_neural_cdes_b200 import _lib
    from perm_equiv_graph_neural_cdes_b200 import dist as pdist

    dev, world, rank = D.dev, D.world, D.rank
    n, h, e, L, T, B = wl["n"], wl["h"], wl["e"], wl["L"], wl["T"], wl["B"]
    flags = operand_flags(args)
    widths_out = 2 * h * e if e > 0 else h
    vf = P.PermEquivGraphVectorField(h, h, widths_out, L, e, n, key=1234, flags=flags).to(dev)
    term = P.ODETerm(P.CDEWrapperVectorField(vf, h) if e > 0 else vf)
    ts, cadj, xco, y0, gy, host, snaps_dev, x_t = make_inputs(wl, 1234 + rank, dev, host_copy=with_e2e, coeff_budget=coeff_budget)
    pc = P.pack_control(ts, cadj, xco) if cadj is not None else P.build_control(ts, snaps_dev, x_t)
    torch.cuda.synchronize()
    del cadj, xco, snaps_dev
    torch.cuda.empty_cache()
    t1_solve = wl.get("t1_solve", wl["t1"])
    step_ts = P.constant_step_table(0.0, t1_solve, wl["dt0"])
    S = len(step_ts) - 1
    l = _lib.lib()
    params = list(vf.parameters())

    def solve_step(pc_, y0_, reduce=True):
        """Returns what a caller of the solve receives: (loss, flat parameter gradient, y(t1), dloss/dy0)."""
        vf.zero_grad(set_to_none=True)
        y = y0_.detach().requires_grad_(True)
        sol = P.diffeqsolve(term, P.Tsit5(), 0.0, t1_solve, wl["dt0"], y, [pc_, None] if e > 0 else pc_,
                            stepsize_controller=P.ConstantStepSize(), saveat=P.SaveAt(t1=True))
        yT = sol.ys[-1]
        loss = (yT * gy).sum()
        loss.backward()
        if reduce:   # ONE all-reduce of the flat parameter-gradient buffer (dist.allreduce_gradients; a no-op at world size 1)
            return loss, pdist.allreduce_gradients(params), yT.detach(), y.grad
        return loss, torch.cat([p.grad.reshape(-1) for p in params]), yT.detach(), y.grad

    for _ in range(max(warmup, 1)):
        solve_step(pc, y0)
    D.barrier()
    graph = None
    l.pegncde_profile_enable(args.profile_stride)
    launches0 = l.pegncde_launch_count()
    if not args.no_graph:
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            solve_step(pc, y0, reduce=False)   # warm the capture stream's workspace
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        l.pegncde_profile_enable(args.profile_stride)
        launches0 = l.pegncde_launch_count()
        with torch.cuda.graph(graph):
            g_out = solve_step(pc, y0, reduce=False)
        launches_per_step = l.pegncde_launch_count() - launches0
        for _ in range(2):
            graph.replay()
        D.barrier()

    def timed_step():
        if graph is not None:
            graph.replay()
            if world > 1:
                torch.distributed.all_reduce(g_out[1])
            return g_out
        return solve_step(pc, y0)

    sampler = ClockSampler(D.local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    host_t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        out = timed_step()
    e1.record()
    host_ms = (time.perf_counter() - host_t0) * 1e3 / steps
    D.barrier()
    clocks = sampler.summary()
    ms = e0.elapsed_time(e1)
    reduced = out[1]
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, dict(zip(("loss", "grad_params", "yT", "grad_y0"), out)))
    # the reduced gradient buffer must be finite and identical on every rank
    grad_check = {"finite": bool(torch.isfinite(reduced).all())}
    if world > 1:
        lo, hi = reduced.clone(), reduced.clone()
        torch.distributed.all_reduce(lo, op=torch.distributed.ReduceOp.MIN)
        torch.distributed.all_reduce(hi, op=torch.distributed.ReduceOp.MAX)
        grad_check["identical_across_ranks"] = bool(torch.equal(lo, hi))
    if (not grad_check["finite"] or grad_check.get("identical_across_ranks") is False) and not os.environ.get("PEG_BENCH_NOCHECK"):
        raise RuntimeError(f"{wl_name}: reduced parameter gradients failed the sanity check {grad_check}")
    if graph is None:
        launches_per_step = (l.pegncde_launch_count() - launches0) // max(steps, 1)
    prof = {}
    for d, nm in ((0, "fwd"), (1, "bwd")):
        a, b_, c_, by, fl = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
        l.pegncde_profile_read(d, a, b_, c_, by, fl)
        prof[nm] = dict(launches=a.value, timed=b_.value, ms=c_.value, bytes=by.value, flops=fl.value)
    l.pegncde_profile_enable(0)
    prof_steps = 1 if graph is not None else steps   # a replayed graph re-records the same event pairs
    ms_per_step = D.max_ms(ms) / steps
    value = world * B * S / (ms_per_step * 1e-3)
    res = {"workload": wl_name, "value": value, "ms_per_step": ms_per_step, "solver_steps": S, "graphs_per_gpu": B, "host_ms_per_step": host_ms,
           "launches": int(launches_per_step * steps), "cuda_graph": graph is not None, "clocks": clocks, "grad_check": grad_check,
           "n_params": int(sum(p.numel() for p in params)), "planes_mb": pc.adj_coef.numel() * 4 / 1e6}

    # ---------------- end-to-end legs: host buffers through the public API ----------------
    if with_e2e:
        d2h = res["n_params"] * 4 + 4

        def e2e_coeff_step():
            # reference-layout coefficient arrays (pinned host memory) -> pack_control keeps them on the host and the solve
            # streams them piece by piece (copy + pack of piece i+1 overlap the steps inside piece i)
            y0_d = host["y0"].to(dev, non_blocking=True)
            pc_ = P.pack_control(host["ts"], host["cadj"], host["xco"], device=dev)
            loss, flat_g = solve_step(pc_, y0_d)[:2]
            return float(loss.item()), flat_g.cpu()

        def e2e_snap_step():
            # one stage earlier (SURVEY N2): graph SNAPSHOTS A_k [B,T,n,n] from the host; Hermite coefficients + tiling on the device
            ts_d = host["ts"].to(dev, non_blocking=True)
            A_d = host["snaps"].to(dev, non_blocking=True)
            x_d = None if host["x_t"] is None else host["x_t"].to(dev, non_blocking=True)
            y0_d = host["y0"].to(dev, non_blocking=True)
            pc_ = P.build_control(ts_d, A_d, x_d)
            loss, flat_g = solve_step(pc_, y0_d)[:2]
            return float(loss.item()), flat_g.cpu()

        def time_leg(fn):
            fn()
            D.barrier()
            e0.record()
            for _ in range(e2e_steps):
                fn()
            e1.record()
            D.barrier()
            return world * B * S / (D.max_ms(e0.elapsed_time(e1)) / e2e_steps * 1e-3)

        base_h2d = host["y0"].numel() * 4 + host["ts"].numel() * 4
        legs = {}
        if host["cadj"] is not None:
            h2d = base_h2d + sum(c.numel() * 4 for c in host["cadj"]) + (sum(c.numel() * 4 for c in host["xco"]) if host["xco"] is not None else 0)
            legs["coefficients"] = {"value": time_leg(e2e_coeff_step), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                                    "input": "reference-layout coefficient arrays (d,c,b,a) [B,T-1,n,n,2] in pinned host memory -> pack_control / diffeqsolve (streamed: copy + pack of cubic piece i+1 overlap the steps inside piece i)"}
        h2d_snap = base_h2d + host["snaps"].numel() * 4 + (0 if host["x_t"] is None else host["x_t"].numel() * 4)
        legs["snapshots"] = {"value": time_leg(e2e_snap_step), "unit": UNIT, "h2d_bytes_per_step": h2d_snap, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                             "input": "graph snapshots A_k [B,T,n,n] in pinned host memory -> build_control (pegncde_build_adj: Hermite coefficients + tiling on the device) / diffeqsolve"}
        res["e2e_legs"] = legs

    # ---------------- roofline of the dominant kernel (the n x n x d contraction) ----------------
    pk = peaks()
    tot_ms = prof["fwd"]["ms"] + prof["bwd"]["ms"]
    tot_timed = prof["fwd"]["timed"] + prof["bwd"]["timed"]
    if tot_timed:
        by = (prof["fwd"]["bytes"] * prof["fwd"]["timed"] + prof["bwd"]["bytes"] * prof["bwd"]["timed"])
        fl = (prof["fwd"]["flops"] * prof["fwd"]["timed"] + prof["bwd"]["flops"] * prof["bwd"]["timed"])
        gbs = by / (tot_ms * 1e-3) / 1e9
        tfs = fl / (tot_ms * 1e-3) / 1e12
        # The planes stream from HBM once per launch; the tensor pipe executes `passes` MMAs per algorithmic product (x = hi + lo
        # split of both operands: hi*hi + lo*hi + hi*lo; 1 with --tf32-fast).  The tensor peak is the cuBLAS GEMM rate of the
        # operand type, measured in this run (tensor_peaks).
        use_tc = bool(flags & 1)
        passes = 1 if (flags & 2) or not use_tc else 3
        fmt = "fp32 FFMA" if not use_tc else ("tf32" if flags & (2 | 8 | 16) else ("bf16" if flags & 32 else "fp16"))
        tpeak = tpeaks.get(fmt) if tpeaks else None
        if tpeak is None:
            tpeak = pk["bf16"] / 2.0 if fmt == "tf32" else pk["bf16"]
        exec_tfs = passes * tfs
        t_hbm, t_tc = by / (pk["hbm"] * 1e9), passes * fl / (tpeak * 1e12)
        bound = "hbm" if t_hbm >= t_tc else "tensor"
        share = tot_ms * (prof["fwd"]["launches"] + prof["bwd"]["launches"]) / max(tot_timed, 1) / (ms_per_step * prof_steps)
        res["roofline"] = {
            "bound": bound, "kernel": "k_tc_contract<fwd> + k_tc_contract<adjoint> (the n x n x d contraction)" if use_tc else "k_dual_contract (FFMA)",
            "achieved": gbs if bound == "hbm" else exec_tfs, "peak": pk["hbm"] if bound == "hbm" else tpeak,
            "unit": "GB/s" if bound == "hbm" else "TFLOP/s", "frac": (gbs / pk["hbm"]) if bound == "hbm" else (exec_tfs / tpeak),
            "peak_source": pk["src"] + " hbm_gbs (MEASURED_PEAKS.json)" if bound == "hbm" else "cuBLAS %s GEMM 8192^3 measured in this run" % fmt,
            "traffic": measured_traffic(wl_name), "achieved_gbs": gbs, "hbm_frac": gbs / pk["hbm"], "algorithmic_tflops": tfs,
            "operand_format": fmt, "tensor_passes": passes, "executed_tflops": exec_tfs, "tensor_peak_tflops": tpeak, "executed_tensor_frac": exec_tfs / tpeak,
            "avg_launch_us": tot_ms / tot_timed * 1e3, "launches_timed": tot_timed, "share_of_step": share,
            "fwd_avg_us": prof["fwd"]["ms"] / max(prof["fwd"]["timed"], 1) * 1e3, "bwd_avg_us": prof["bwd"]["ms"] / max(prof["bwd"]["timed"], 1) * 1e3,
            "fwd_gbs": prof["fwd"]["bytes"] * prof["fwd"]["timed"] / max(prof["fwd"]["ms"], 1e-9) / 1e6,
            "bwd_gbs": prof["bwd"]["bytes"] * prof["bwd"]["timed"] / max(prof["bwd"]["ms"], 1e-9) / 1e6,
            "algorithmic_bytes_per_launch": {"fwd": prof["fwd"]["bytes"], "adjoint": prof["bwd"]["bytes"]},
            "algorithmic_flops_per_launch": {"fwd": prof["fwd"]["flops"], "adjoint": prof["bwd"]["flops"]},
            "whole_step_gbs": (prof["fwd"]["bytes"] * prof["fwd"]["launches"] + prof["bwd"]["bytes"] * prof["bwd"]["launches"]) / prof_steps / (ms_per_step * 1e-3) / 1e9,
            "l2_note": "planes %s L2 (126 MB)" % ("fit in" if 16.0 * n * n * B <= 126e6 else "exceed")}
    else:
        res["roofline"] = None
    del pc, vf, graph
    torch.cuda.empty_cache()
    return res


def measure_heat(D, args, steps, warmup):
    """BASELINE.json configs[0]: the dynamical-systems default (perm_equiv_gncde_config.yaml): heat diffusion on n = 400 nodes, B = 4
    trajectories, h = 16, L = 2, Tsit5 + PIDController(1e-3, 1e-6), dt0 = None, SaveAt(ts = ts) (dense output at the 20 knots),
    forward + exact adjoint over the accepted steps.  value = attempted solver steps of all trajectories per second."""
    import perm_equiv_graph_neural_cdes_b200 as P

    dev = D.dev
    n, h, L, T, B = 400, 16, 2, 20, 4
    g = torch.Generator(device=dev).manual_seed(99 + D.rank)
    ts = torch.linspace(0.0, 5.0, T, device=dev)
    A = torch.stack([synth_adjacency(n, T, 700 + 10 * D.rank + b, dev) for b in range(B)])
    vf = P.PermEquivGraphVectorField(h, h, h, L, 0, n, key=1234, flags=operand_flags(args)).to(dev)
    pc = P.build_control(ts, A)
    y0 = torch.randn((B, n, h), generator=g, device=dev)
    params = list(vf.parameters())
    from perm_equiv_graph_neural_cdes_b200 import dist as pdist

    def step():
        vf.zero_grad(set_to_none=True)
        y = y0.detach().requires_grad_(True)
        sol = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 5.0, None, y, pc, stepsize_controller=P.PIDController(rtol=1e-3, atol=1e-6), saveat=P.SaveAt(ts=ts))
        sol.ys.square().mean().backward()
        pdist.allreduce_gradients(params)
        st = sol.stats["num_steps"]
        return int(sum(st)) if isinstance(st, (list, tuple)) else int(st) * B

    for _ in range(max(warmup, 1)):
        attempted = step()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        attempted = step()
    e1.record()
    D.barrier()
    ms = D.max_ms(e0.elapsed_time(e1)) / steps
    return {"workload": "heat (configs[0]: n=400, B=4, h=16, L=2, adaptive Tsit5 rtol 1e-3, SaveAt(ts))", "value": D.world * attempted / (ms * 1e-3), "unit": UNIT,
            "ms_per_step": ms, "attempted_solver_steps_per_gpu": attempted, "graphs_per_gpu": B,
            "note": "adaptive path: the whole batch steps per launch with per-trajectory (t, dt) on the device (pegncde_step_fwd_batched + pegncde_adaptive_control); the host polls the done flags every 8 attempts"}


def run_ours(args):
    import perm_equiv_graph_neural_cdes_b200 as P  # noqa: F401  (raises if libpegncde.so is missing: no CPU fallback)

    D = Dist()
    wl = dict(WORKLOADS[args.workload])
    if args.batch:
        wl["B"] = args.batch
    if args.t1 > 0:
        wl["t1_solve"] = args.t1
    tpeaks = None if args.no_tensor_peaks else tensor_peaks(D.dev)
    head = measure_fixed(D, args.workload, wl, args, args.steps, args.warmup, with_e2e=True, tpeaks=tpeaks,
                         e2e_steps=max(1, min(args.steps, args.e2e_steps)), dump_dir=args.dump_outputs)

    # ---- the other points of BASELINE.json configs[4] (short solves: t1 = 0.5 -> 5 solver steps, T = 3 knots) and configs[0..3] ----
    sweep, configs = [], []
    if not args.no_sweep:
        for name in SWEEP_POINTS:
            w2 = dict(WORKLOADS[name], T=3, t1=2.0, t1_solve=0.5)
            r = measure_fixed(D, name, w2, args, 2, 3, with_e2e=True, tpeaks=tpeaks, e2e_steps=1, coeff_budget=0)   # snapshots only
            rf = r["roofline"] or {}
            sweep.append({"workload": name, "n": w2["n"], "hidden": w2["h"], "data_embed_dim": w2["e"], "graphs_per_gpu": w2["B"], "solver_steps": r["solver_steps"],
                          "value": r["value"], "unit": UNIT, "frac": rf.get("frac"), "bound": rf.get("bound"), "hbm_frac": rf.get("hbm_frac"),
                          "executed_tensor_frac": rf.get("executed_tensor_frac"), "fwd_gbs": rf.get("fwd_gbs"), "bwd_gbs": rf.get("bwd_gbs"),
                          "share_of_step": rf.get("share_of_step"), "e2e": r["e2e_legs"]["snapshots"]["value"],
                          "e2e_input": "graph snapshots from pinned host memory", "note": "short solve: 3 knots, t1 = 0.5 (5 solver steps), 2 timed steps"})
        for name in ("sir", "england", "twitter"):
            r = measure_fixed(D, name, dict(WORKLOADS[name]), args, 3, 3, with_e2e=True, tpeaks=tpeaks, e2e_steps=1)
            legs = r["e2e_legs"]
            configs.append({"workload": name, "config": CONFIG_OF[name], "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "graphs_per_gpu": r["graphs_per_gpu"],
                            "solver_steps": r["solver_steps"], "e2e": max(v["value"] for v in legs.values()), "cuda_graph": r["cuda_graph"],
                            "frac": (r["roofline"] or {}).get("frac")})
        heat = dict(measure_heat(D, args, 2, 1), config="configs[0]")
        if D.rank == 0 and D.world == 1 and not args.no_cpu_baseline:
            heat["cpu_baseline"] = cpu_baseline_heat()
        configs.insert(0, heat)

    cpu_base = None
    if D.rank == 0 and D.world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_baseline(wl, args)

    if D.rank == 0:
        n, h, e, L, T, B = wl["n"], wl["h"], wl["e"], wl["L"], wl["T"], wl["B"]
        flags = operand_flags(args)
        legs = head["e2e_legs"]
        best = max(legs, key=lambda k: legs[k]["value"])   # the headline end-to-end number is the faster public entry point; both are reported
        fmt = (head["roofline"] or {}).get("operand_format", "fp32 FFMA")
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (n x n x d contraction on tcgen05: %s split operands, three products, fp32 accumulate)" % fmt if flags & 1 and not flags & 2 else
                     ("f32 (contraction: 1xTF32 tcgen05)" if flags & 2 else "f32 (CUDA-core FFMA)"),
            "data": "synthetic",
            "config": {"workload": args.workload, "n": n, "hidden": h, "data_embed_dim": e, "layers": L, "knots": T,
                       "solver": "Tsit5 fixed dt0=%g" % wl["dt0"], "solver_steps": head["solver_steps"], "graphs_per_gpu": B,
                       "parallelism": "batch of trajectories sharded over %d GPU(s); NCCL all-reduce of %d param grads" % (D.world, head["n_params"]),
                       "l2": "inputs per GPU %.0f MB of coefficient planes (> L2 126 MB: %s)" % (head["planes_mb"], head["planes_mb"] * 1e6 > 126e6)},
            "e2e": dict(legs[best], entry=best),
            "e2e_from_coefficients": legs.get("coefficients"), "e2e_from_snapshots": legs.get("snapshots"),
            "gpu_launches": head["launches"], "cuda_graph": head["cuda_graph"], "host_ms_per_step": head["host_ms_per_step"], "clocks": head["clocks"],
            "grad_check": head["grad_check"], "tensor_peaks_tflops": tpeaks, "roofline": head["roofline"], "cpu_baseline": cpu_base,
            "sweep": sweep, "configs": configs,
        }
        print(json.dumps(line))
    if D.world > 1:
        torch.distributed.destroy_process_group()


def hashed_strip(n, rows, T, seed, device, transposed):
    """Synthetic dynamic weighted digraph given ELEMENTWISE by a hash of (knot, i, j), so that every rank can build exactly its strip:
    `rows` = (r0, r1); returns A_k[:, r0:r1, :] as [T, r1-r0, n], or with transposed=True the same rows of the transposed path
    (A_k[:, :, r0:r1] transposed).  ~16 weighted out-edges per node, unit self-loops, entries drifting slowly from knot to knot."""
    r0, r1 = rows
    a = torch.arange(r0, r1, device=device, dtype=torch.float32)[:, None]
    b = torch.arange(n, device=device, dtype=torch.float32)[None, :]
    i, j = (b, a) if transposed else (a, b)       # element (i, j) of the path sits at [i - r0, j], of the transposed strip at [j - r0, i]
    def h(k1, k2, k3):
        return torch.frac(torch.sin(i * k1 + j * k2 + (seed % 97) * k3) * 43758.5453).abs()
    mask = (h(12.9898, 78.233, 37.719) < 16.0 / n).to(torch.float32)
    w0, w1 = 0.25 + h(4.898, 7.23, 1.17), h(9.12, 3.77, 2.31) - 0.5
    eye = (i == j).to(torch.float32)
    out = torch.empty((T, r1 - r0, n), device=device)
    for k in range(T):
        out[k] = (mask * (w0 + 0.15 * k * w1) + eye) / 16.0
    return out


def run_rowsharded(args):
    """`--shard rows`: ONE graph trajectory of the workload spread over the ranks by rows (BASELINE.json configs[4] "row-sharded A at
    largest n"), forward + exact adjoint; the per-layer exchange of V^T runs over peer memory (k_shard_push / k_shard_wait)."""
    import perm_equiv_graph_neural_cdes_b200 as P
    from perm_equiv_graph_neural_cdes_b200 import _lib, rowshard as RS

    D = Dist()
    wl = dict(WORKLOADS[args.workload])
    n, h, L = wl["n"], wl["h"], wl["L"]
    if wl["e"] != 0:
        raise SystemExit("--shard rows: workloads without the CDE wrapper (e = 0)")
    B = args.batch or 1
    T, t1 = 3, 2.0
    t1_solve = args.t1 if args.t1 > 0 else 1.0
    dev = D.dev
    flags = operand_flags(args)
    r0, r1 = RS.row_range(n, D.rank, D.world)
    ts = torch.arange(T, device=dev, dtype=torch.float32) * (t1 / (T - 1))
    rows = torch.stack([hashed_strip(n, (r0, r1), T, 1234 + b, dev, False) for b in range(B)])
    cols = torch.stack([hashed_strip(n, (r0, r1), T, 1234 + b, dev, True) for b in range(B)])
    ctl = RS.RowShardedControl(ts, rows, cols, h, L, flags=flags)
    del rows, cols
    torch.cuda.empty_cache()
    vf = P.PermEquivGraphVectorField(h, h, h, L, 0, n, key=1234, flags=flags).to(dev)
    g = torch.Generator(device=dev).manual_seed(77)           # the same full state on every rank, each keeps its rows
    y0 = torch.randn((B, n, h), generator=g, device=dev)[:, r0:r1].contiguous()
    gy = torch.randn((B, n, h), generator=g, device=dev)[:, r0:r1].contiguous()
    S = len(P.constant_step_table(0.0, t1_solve, wl["dt0"])) - 1
    l = _lib.lib()

    def step(reduce=True):
        vf.zero_grad(set_to_none=True)
        y = y0.detach().requires_grad_(True)
        yT = RS.diffeqsolve_rowsharded(vf, ctl, y, 0.0, t1_solve, wl["dt0"], reduce_grads=False)
        (yT * gy).sum().backward()
        flat_ = torch.cat([p.grad.reshape(-1) for p in vf.parameters()])
        if reduce and D.world > 1:      # per-rank partial sums over the rank's rows -> the parameter gradient
            torch.distributed.all_reduce(flat_)
        return flat_

    for _ in range(max(args.warmup, 1)):
        flat = step()
    D.barrier()
    # the whole step (forward + adjoint, exchanges included: device-side epoch base) replays as ONE CUDA graph; the all-reduce of
    # the flat gradient buffer stays outside, as in the batch-sharded path
    graph = None
    l.pegncde_profile_enable(args.profile_stride)
    launches0 = l.pegncde_launch_count()
    if not args.no_graph:
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step(reduce=False)          # warm the capture stream's workspace
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        D.barrier()
        l.pegncde_profile_enable(args.profile_stride)
        launches0 = l.pegncde_launch_count()
        with torch.cuda.graph(graph):
            g_flat = step(reduce=False)
        launches_per_step = l.pegncde_launch_count() - launches0
        for _ in range(2):
            graph.replay()
        D.barrier()

    def timed_step():
        if graph is not None:
            graph.replay()
            if D.world > 1:
                torch.distributed.all_reduce(g_flat)
            return g_flat
        return step()

    sampler = ClockSampler(D.local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        flat = timed_step()
    e1.record()
    D.barrier()
    clocks = sampler.summary()
    ms_per_step = D.max_ms(e0.elapsed_time(e1)) / args.steps
    launches = launches_per_step * args.steps if graph is not None else l.pegncde_launch_count() - launches0
    prof = {}
    for d_, nm in ((0, "fwd"), (1, "bwd")):
        a, b_, c_, by, fl = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
        l.pegncde_profile_read(d_, a, b_, c_, by, fl)
        prof[nm] = dict(launches=a.value, timed=b_.value, ms=c_.value)
    l.pegncde_profile_enable(0)
    lo, hi = flat.clone(), flat.clone()
    if D.world > 1:
        torch.distributed.all_reduce(lo, op=torch.distributed.ReduceOp.MIN)
        torch.distributed.all_reduce(hi, op=torch.distributed.ReduceOp.MAX)
    grad_check = {"finite": bool(torch.isfinite(flat).all()), "identical_across_ranks": bool(torch.equal(lo, hi))}
    if D.rank == 0:
        pk = peaks()
        nloc = r1 - r0
        # per contraction launch and rank: the strip of the path AND the strip of its transpose stream from HBM once (2 x 16 nloc n B);
        # the exchange ships this rank's slice of V^T (hi + lo parts) to every peer
        esz = 4 if args.operands == "tf32x3" else 2
        bytes_launch = B * 2 * 16.0 * nloc * n
        tot_ms = prof["fwd"]["ms"] + prof["bwd"]["ms"]
        tot_timed = prof["fwd"]["timed"] + prof["bwd"]["timed"]
        gbs = bytes_launch * tot_timed / max(tot_ms, 1e-9) / 1e6
        exchanges = S * (6 + 6) * L + S * 0
        nvlink = (D.world - 1) * B * h * nloc * esz * 2
        line = {"metric": METRIC, "value": B * S / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32 (contraction: %s split operands on tcgen05, fp32 accumulate)" % args.operands, "data": "synthetic",
                "config": {"workload": args.workload, "shard": "rows", "n": n, "hidden": h, "layers": L, "knots": T, "graphs": B, "solver_steps": S,
                           "rows_per_gpu": nloc, "parallelism": "ONE graph row-sharded over %d GPU(s): strips of the path and of its transpose per rank; V^T exchanged per layer over peer memory (k_shard_push / k_shard_wait), parameter gradients all-reduced (NCCL)" % D.world},
                "gpu_launches": int(launches), "cuda_graph": graph is not None, "clocks": clocks, "grad_check": grad_check,
                "exchange": {"per_solver_step": 12 * L, "nvlink_bytes_per_exchange_and_rank": nvlink, "nvlink_bytes_per_step_and_rank": nvlink * exchanges},
                "roofline": {"bound": "hbm", "kernel": "k_tc_contract (row strips)", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                             "traffic": None, "algorithmic_bytes_per_launch": bytes_launch, "fwd_avg_us": prof["fwd"]["ms"] / max(prof["fwd"]["timed"], 1) * 1e3,
                             "bwd_avg_us": prof["bwd"]["ms"] / max(prof["bwd"]["timed"], 1) * 1e3,
                             "note": "timed region of a launch = conversion of V (top adjoint layer only) + exchange (push, wait) + contraction"}}
        print(json.dumps(line))
    if D.world > 1:
        torch.distributed.destroy_process_group()


# points of BASELINE.json configs[4] reported in the `sweep` array of every run (n in {1k, 4k, 16k} x h in {64, 256} + the wide last layer)
SWEEP_POINTS = ["sweep_n1024_h64", "sweep_n1024_h256", "sweep_n4096_h64", "sweep_n4096_h256", "sweep_n16384_h64", "sweep_n16384_h256", "sweep_n1024_h128_e8"]
CONFIG_OF = {"sir": "configs[1] (SIR, n=100, B=50 per GPU)", "england": "configs[2] (PGT England shape, n=129)", "twitter": "configs[3] (PGT Twitter shape, n=1000, e=16)"}


def cpu_problem(wl, seed, sample_steps):
    """The same workload shape for the CPU oracle, restricted to the first `sample_steps` solver steps."""
    from oracle import reference_path as R

    p = R.make_problem(n=wl["n"], h=wl["h"], e=wl["e"], L=wl["L"], T=wl["T"], t1=wl["t1"], dt0=wl["dt0"], seed=seed,
                       float_ts=bool(wl.get("float_ts")), randomize_norm=False)
    p.step_ts = p.step_ts[: sample_steps + 1]
    return p


def oracle_segments(wl, sample_steps):
    """The CPU sample as (segment length, count): autograd through one solve keeps every stage's materialised n x n adjacency, so
    at n >= 1024 the sample runs as independent solves of at most 6 steps (same arithmetic per step, bounded host memory)."""
    seg = min(sample_steps, 6) if wl["n"] >= 1024 else sample_steps
    return seg, max(1, sample_steps // seg)


def run_oracle_sample(wl, sample_steps):
    """Seconds for `segments x seg` solver steps forward + backward of the oracle; returns (steps done, seconds)."""
    from oracle import reference_path as R

    seg, cnt = oracle_segments(wl, sample_steps)
    p = cpu_problem(wl, 1234, seg)
    t0 = time.perf_counter()
    for _ in range(cnt):
        R.run_forward_backward(p)
    return seg * cnt, time.perf_counter() - t0


def time_oracle(wl, sample_steps, repeats, threads):
    from oracle import reference_path as R

    torch.set_num_threads(threads)
    R.run_forward_backward(cpu_problem(wl, 1234, 1))  # warm-up
    done, dt = 0, 0.0
    for _ in range(repeats):
        k, t = run_oracle_sample(wl, sample_steps)
        done += k
        dt += t
    return done / dt, dt / repeats


def cpu_baseline(wl, args):
    threads = os.cpu_count() or 1
    sample_steps = args.cpu_sample_steps
    v, dt = time_oracle(wl, sample_steps, 1, threads)
    return {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "1 graph x %d solver steps fwd+bwd of the same workload shape (%d solve(s) of %d steps), torch-CPU restatement (oracle), %.1f s"
                      % ((lambda sc: (sc[0] * sc[1], sc[1], sc[0]))(oracle_segments(wl, sample_steps)) + (dt,))}


def cpu_baseline_heat():
    """The heat configuration (configs[0]) on the host cores: ONE trajectory of the restated adaptive solve (oracle), forward + autograd
    backward, timed once after a short warm-up; value = attempted solver steps per second."""
    import numpy as np

    from oracle import reference_path as R

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    n, h, L, T = 400, 16, 2, 20
    p = R.make_problem(n=n, h=h, e=0, L=L, T=T, t1=5.0, dt0=0.1, seed=99, float_ts=True, randomize_norm=False)

    def run():
        layers = R.params_to(p.layers, requires_grad=True)
        y0 = p.y0.clone().requires_grad_(True)
        ca = R.CubicInterpolation(p.ts, p.coeffs_adj)
        f = lambda t, y: R.perm_equiv_vector_field(t, y, ca, layers)
        ys, table, stats = R.tsit5_solve_adaptive(f, y0, float(p.ts[0]), float(p.ts[-1]), rtol=1e-3, atol=1e-6, dt0=None, save_ts=[float(t) for t in p.ts])
        ys.square().mean().backward()
        return int(stats["num_steps"])

    run()
    t0 = time.perf_counter()
    attempts = run()
    dt = time.perf_counter() - t0
    return {"value": attempts / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "1 trajectory (n=400, h=16, L=2) adaptive fwd+bwd, torch-CPU restatement (oracle), %d attempted steps in %.1f s" % (attempts, dt)}


def run_reference(args):
    """Reference arm: the reference's own CPU algorithm (the oracle port -- JAX/diffrax are not installable here)
    with all host threads on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = dict(WORKLOADS[args.workload])
    threads = os.cpu_count() or 1
    from oracle import reference_path as R

    torch.set_num_threads(threads)
    seg, cnt = oracle_segments(wl, args.cpu_sample_steps)
    sample_steps = seg * cnt
    for _ in range(min(args.warmup, 1)):
        R.run_forward_backward(cpu_problem(wl, 1234, 1))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run_oracle_sample(wl, args.cpu_sample_steps)
    dt = (time.perf_counter() - t0) / args.steps
    v = sample_steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "n": wl["n"], "hidden": wl["h"], "data_embed_dim": wl["e"], "layers": wl["L"],
                       "knots": wl["T"], "solver": "Tsit5 fixed dt0=%g" % wl["dt0"],
                       "solver_steps": len(R.constant_step_table(0.0, wl["t1"], wl["dt0"])) - 1, "graphs_per_gpu": wl["B"],
                       "parallelism": "host threads of one box (the reference has no multi-device path)"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "each step = 1 graph x %d solver steps fwd+bwd in %d solve(s) of %d steps (torch-CPU restatement of the reference path)" % (sample_steps, cnt, seg)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="graphs per GPU (default: the workload's)")
    ap.add_argument("--no-tensor-cores", action="store_true")
    ap.add_argument("--tf32-fast", action="store_true")
    ap.add_argument("--operands", default="fp16x2", choices=["fp16x2", "bf16x2", "tf32x3"],
                    help="operand format of the tcgen05 contraction: fp16x2 with block exponents (default), bf16x2 (looser tolerance), 3xTF32")
    ap.add_argument("--profile-stride", type=int, default=4)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-sample-steps", type=int, default=24, help="solver steps of one graph the CPU baseline runs (~15 s of CPU work at the default workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from the host instead of replaying a CUDA graph")
    ap.add_argument("--t1", type=float, default=0.0, help="profiling only: shorten the solve to [0, t1] (fewer solver steps)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the `sweep` / `configs` arrays (the other BASELINE.json configurations)")
    ap.add_argument("--no-tensor-peaks", action="store_true", help="skip the live cuBLAS tf32 / fp16 / bf16 GEMM measurement")
    ap.add_argument("--shard", default="batch", choices=["batch", "rows"],
                    help="batch: trajectories sharded over the GPUs (default); rows: ONE graph row-sharded over the GPUs (large n)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (loss, flat parameter gradient, y(t1), dloss/dy0; "
                         "rank 0's shard) as DIR/<name>.npy in float32, at most 64 MB in all (a fixed, seeded sample past that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.shard != "batch"):
        ap.error("--dump-outputs writes the outputs of the batch-sharded CUDA path (--impl ours --shard batch)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "ours" and args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        # `python bench.py --gpus N` outside torchrun: launch the ranks ourselves (one per GPU, NCCL, loopback rendezvous)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 2000), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if world > 1 and args.gpus not in (1, world):
        raise SystemExit(f"--gpus {args.gpus} contradicts WORLD_SIZE={world}")
    if args.impl == "reference":
        run_reference(args)
    elif args.shard == "rows":
        run_rowsharded(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
