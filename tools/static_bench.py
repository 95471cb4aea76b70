"""Static controls against the replicated dense control on the benchmark's shapes: prints ONE JSON line.

  python tools/static_bench.py [--steps K] [--warmup W] [--rounds R] [--workloads a,b,...] [--out FILE]

A static control (build_static_control) stores one plane per graph; the replicated control (build_control on the snapshots
[A] * T) stores four planes per piece with b = c = d = 0.  Both compute the same y(T) and dloss/dy0 bit for bit, which this tool
asserts for one eager forward + exact-adjoint solve; the parameter gradient (float-atomic reductions) is reported and checked to 1e-5.  For every workload, with the two legs
alternated `rounds` times in one process: solver steps/s of forward + adjoint (CUDA-graph replay, as bench.py), and -- in a
torch.profiler run of its own -- the device microseconds per launch of the forward and adjoint contraction, their algorithmic
bytes over that time (the profiling hooks' count: planes + V + OUT (+ M)) and the share of the copy bandwidth measured on a
B200 (COPY_GBPS).  static_n65536_h128 has no dense leg: its 16 n^2 bytes per piece would not fit in device memory.
The GPU name, power limit and SM clocks are read in the same call.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
import perm_equiv_graph_neural_cdes_b200 as P  # noqa: E402
from perm_equiv_graph_neural_cdes_b200 import _lib  # noqa: E402

WORKLOADS = {
    "sweep_n2048_h128": dict(bench.WORKLOADS["sweep_n2048_h128"]),
    "sweep_n16384_h128": dict(bench.WORKLOADS["sweep_n16384_h128"]),
    # capacity point: one plane of 17.2 GB; a dense control would need 68.7 GB per piece.  Eight steps keep the run short.
    "static_n65536_h128": dict(n=65536, h=128, e=0, L=3, T=9, t1=8.0, dt0=1.0, B=1, dense=False),
}
COPY_GBPS = 6549.1     # HBM copy bandwidth measured on a B200 (DESIGN.md, "Measured"): the bound the contraction is compared with


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True,
                         text=True, timeout=10).stdout.strip()
    name, plim, sm, smax = [x.strip() for x in out.split(",")]
    return dict(name=name, power_limit_w=float(plim), sm_mhz=float(sm), sm_max_mhz=float(smax))


def kernel_us(step, ctl, fwd_pat, bwd_pat):
    """device microseconds per launch of the forward / adjoint contraction in one eager step, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(ctl)
        torch.cuda.synchronize()
    out = {}
    for key, pat in (("fwd", fwd_pat), ("bwd", bwd_pat)):
        evs = [e for e in prof.key_averages() if pat in e.key]
        cnt = sum(e.count for e in evs)
        tot = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in evs)
        out[key] = dict(launches=cnt, us_per_launch=tot / max(cnt, 1))
    return out


def hook_bytes(lib, step, ctl):
    """algorithmic bytes of one forward / adjoint contraction launch (pegncde_profile_read)"""
    lib.pegncde_profile_enable(1)
    step(ctl)
    torch.cuda.synchronize()
    out = {}
    for d, nm in ((0, "fwd"), (1, "bwd")):
        a, t_, ms, by, fl = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
        lib.pegncde_profile_read(d, a, t_, ms, by, fl)
        out[nm] = by.value
    lib.pegncde_profile_enable(0)
    return out


def measure(name, wl, steps, warmup, rounds, dev):
    n, h, L, T, B = wl["n"], wl["h"], wl["L"], wl["T"], wl["B"]
    ts = torch.arange(T, device=dev, dtype=torch.float32) * (wl["t1"] / (T - 1))
    A = torch.cat([bench.synth_adjacency(n, 1, 4321 * 1000 + b, dev) for b in range(B)])      # [B, n, n]: knot 0 of each graph
    legs = {"static": P.build_static_control(ts, A)}
    if wl.get("dense", True):
        legs["dense"] = P.build_control(ts, A[:, None].expand(B, T, n, n).contiguous())
    del A
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    vf = P.PermEquivGraphVectorField(h, h, h, L, 0, n, key=4321).to(dev)
    params = list(vf.parameters())
    g = torch.Generator(device=dev).manual_seed(4321 + 77)
    y0, gy = torch.randn((B, n, h), generator=g, device=dev), torch.randn((B, n, h), generator=g, device=dev)
    S = len(P.constant_step_table(0.0, wl["t1"], wl["dt0"])) - 1
    lib = _lib.lib()

    def step(ctl):
        for q in params:
            q.grad = None
        y = y0.detach().requires_grad_(True)
        yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, wl["t1"], wl["dt0"], y, ctl, stepsize_controller=P.ConstantStepSize(),
                           saveat=P.SaveAt(t1=True)).ys[-1]
        (yT * gy).sum().backward()
        return yT.detach(), y.grad, torch.cat([q.grad.reshape(-1) for q in params])

    out = dict(workload=name, n=n, h=h, L=L, T=T, B=B, solver_steps=S, static_plane_bytes=legs["static"].adj_static.numel() * 4,
               dense_plane_bytes=(legs["dense"].adj_coef.numel() * 4 if "dense" in legs else B * (T - 1) * 16.0 * legs["static"].ldn ** 2))
    eager = {k: tuple(x.clone() for x in step(c)) for k, c in legs.items()}
    if "dense" in legs:
        same = [bool(torch.equal(a, b)) for a, b in zip(eager["static"], eager["dense"])]
        out["outputs_bit_identical"] = dict(yT=same[0], grad_y0=same[1], grad_params=same[2])
        # the parameter gradient is a float-atomic reduction whose order follows CTA timing (DESIGN.md, "Static controls")
        gs, gd = eager["static"][2].double(), eager["dense"][2].double()
        out["grad_params_max_rel_diff"] = float((gs - gd).abs().max() / gd.abs().max().clamp_min(1e-30))
        assert same[0] and same[1], f"{name}: static and replicated controls differ: {out['outputs_bit_identical']}"
        assert out["grad_params_max_rel_diff"] < 1e-5, out["grad_params_max_rel_diff"]
    else:
        out["finite"] = bool(all(torch.isfinite(x).all() for x in eager["static"]))
        assert out["finite"], name
    del eager
    graphs = {}
    for k, c in legs.items():
        for _ in range(max(warmup, 1)):
            step(c)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step(c)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            step(c)
        gr.replay()
        torch.cuda.synchronize()
        graphs[k] = gr
    ms = {k: [] for k in legs}
    for _ in range(rounds):                       # the legs alternate
        for k in legs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                graphs[k].replay()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / steps)
    del graphs
    for k, c in legs.items():
        fmt = "2, true>" if k == "static" else "2, false>"    # fp16x2 instantiations of k_tc_contract
        kus = kernel_us(step, c, "k_tc_contract<0, " + fmt, "k_tc_contract<1, " + fmt)
        by = hook_bytes(lib, step, c)
        for d in ("fwd", "bwd"):
            us = kus[d]["us_per_launch"]
            kus[d]["bytes_per_launch"] = by[d]
            kus[d]["gbps"] = by[d] / (us * 1e-6) / 1e9 if us > 0 else None
            kus[d]["share_of_copy_bw"] = kus[d]["gbps"] / COPY_GBPS if us > 0 else None
        best = min(ms[k])
        out[k] = dict(ms_per_step_rounds=ms[k], steps_per_s=B * S / (best * 1e-3), contraction=kus)
    if "dense" in legs:
        out["static_over_dense_steps_per_s"] = out["static"]["steps_per_s"] / out["dense"]["steps_per_s"]
        out["static_over_dense_fwd_launch"] = out["dense"]["contraction"]["fwd"]["us_per_launch"] / out["static"]["contraction"]["fwd"]["us_per_launch"]
        out["static_over_dense_bwd_launch"] = out["dense"]["contraction"]["bwd"]["us_per_launch"] / out["static"]["contraction"]["bwd"]["us_per_launch"]
    del legs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.rounds < 1:
        ap.error("--steps and --rounds must be >= 1")
    dev = torch.device("cuda:0")
    info = gpu_info()
    rows = [measure(nm, WORKLOADS[nm], args.steps, args.warmup, args.rounds, dev) for nm in args.workloads.split(",")]
    line = json.dumps(dict(gpu=info, sm_mhz_after=gpu_info()["sm_mhz"], copy_gbps_reference=COPY_GBPS, steps=args.steps,
                           warmup=args.warmup, rounds=args.rounds, workloads=rows))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
