"""Dense planes against sparse (CSR) controls on the benchmark's inputs: prints ONE JSON line.

  python tools/sparse_bench.py [--steps K] [--warmup W] [--workloads a,b,...] [--edge-grads]

The graphs come from bench.py's generator (synth_adjacency); the edge list of a graph is the union of its nonzeros over the
knots, the edge weights are the snapshot values on it.  For every workload: solver steps/s of forward + adjoint (CUDA-graph replay,
as bench.py) on the dense control (build_control) and on the sparse one (build_sparse_control), the contraction's microseconds per
launch from the profiling hooks, nnz per row, HBM bytes per launch (the hooks' algorithmic count) and the V-gather bytes of the
sparse contraction (2 nnz d 4, mostly served from L2), and the largest relative difference of y(T), dloss/dy0 and the parameter
gradient between the two controls.  sparse_n65536_h128 has no dense leg: its planes would not fit in device memory.

--edge-grads adds a sparse leg whose coefficients require grad (a leaf in place of the builder's output, so every replayed step
differentiates the solve w.r.t. them: pegncde_solve_bwd_adj; the once-per-batch Hermite transpose is not part of a step), its ratio
to the plain sparse leg, and the device time per launch of k_sparse_adj_grad (+ its per-node kernels) against k_sparse_contract<4>
from torch.profiler in one eager step of its own.
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
    "sparse_n65536_h128": dict(n=65536, h=128, e=0, L=3, T=9, t1=8.0, dt0=0.1, B=1, dense=False),
}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True,
                             text=True, timeout=10).stdout.strip()
        name, plim, sm, smax = [x.strip() for x in out.split(",")]
        return dict(name=name, power_limit_w=float(plim), sm_mhz=float(sm), sm_max_mhz=float(smax))
    except Exception as ex:   # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), error=str(ex))


def large_path(n, T, seed, device, deg=16):
    """bench.synth_adjacency's statistics without the n x n mask: ~deg random edges per row (Bernoulli(16/n) per entry in the
    generator), a unit self-loop, LogNormal weights, 10 % of the entries redrawn per knot (absent after a redraw with the same
    odds as in the generator, i.e. almost always), rows normalised.  Returns (edge_index, edge_weight [T, E])."""
    g = torch.Generator(device=device).manual_seed(seed)
    rows = torch.cat([torch.arange(n, device=device).repeat_interleave(deg), torch.arange(n, device=device)])
    cols = torch.cat([torch.randint(0, n, (n * deg,), generator=g, device=device), torch.arange(n, device=device)])
    E = rows.numel()
    mask = torch.ones(E, dtype=torch.bool, device=device)
    w = torch.exp(torch.randn(E, generator=g, device=device))
    out = []
    for k in range(T):
        if k > 0:   # a redrawn entry of the generator is a fresh Bernoulli(16/n) draw: the old edge goes, an edge elsewhere comes
            redraw = torch.rand(E, generator=g, device=device) < 0.10
            mask = mask & ~redraw
            w = torch.where(redraw, torch.exp(torch.randn(E, generator=g, device=device)), w)
        wk = torch.where(rows == cols, torch.ones_like(w), torch.where(mask, w, torch.zeros_like(w)))
        out.append(wk / torch.zeros(n, device=device).index_add_(0, rows, wk)[rows])
    return torch.stack([rows, cols]), torch.stack(out)


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def kernel_times(step, pc):
    """device microseconds per launch of the adjoint's sparse kernels in one eager step, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(pc)
        torch.cuda.synchronize()
    out = {}
    for key, pat in (("contract_bwd", "k_sparse_contract<4>"), ("adj_grad", "k_sparse_adj_grad"), ("adj_node", "k_sparse_adj_node"),
                     ("adj_tot", "k_sparse_adj_tot")):
        evs = [e for e in prof.key_averages() if pat in e.key]
        cnt = sum(e.count for e in evs)
        tot = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in evs)
        out[key] = dict(launches=cnt, us_per_launch=tot / max(cnt, 1))
    return out


def measure(name, wl, steps, warmup, dev, edge_grads=False):
    n, h, L, T, B = wl["n"], wl["h"], wl["L"], wl["T"], wl["B"]
    ts = torch.arange(T, device=dev, dtype=torch.float32) * (wl["t1"] / (T - 1))
    with_dense = wl.get("dense", True)
    dense, eis, ews = None, [], []
    if with_dense:
        A = torch.stack([bench.synth_adjacency(n, T, 1234 * 1000 + b, dev) for b in range(B)])
        for b in range(B):
            nz = (A[b] != 0).any(dim=0)
            ei = torch.nonzero(nz).t().contiguous()
            eis.append(ei)
            ews.append(A[b][:, ei[0], ei[1]].contiguous())
        dense = P.build_control(ts, A)
        del A
    else:
        for b in range(B):
            ei, w = large_path(n, T, 1234 * 1000 + b, dev)
            eis.append(ei)
            ews.append(w)
    sparse = P.build_sparse_control(ts, eis, ews, n)
    del eis, ews
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    vf = P.PermEquivGraphVectorField(h, h, h, L, 0, n, key=1234).to(dev)
    params = list(vf.parameters())
    g = torch.Generator(device=dev).manual_seed(1234 + 77)
    y0, gy = torch.randn((B, n, h), generator=g, device=dev), torch.randn((B, n, h), generator=g, device=dev)
    S = len(P.constant_step_table(0.0, wl["t1"], wl["dt0"])) - 1
    lib = _lib.lib()

    def step(pc):
        for q in params:
            q.grad = None
        if pc.adj_packed is not None:
            pc.adj_packed.grad = None
        y = y0.detach().requires_grad_(True)
        yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, wl["t1"], wl["dt0"], y, pc, stepsize_controller=P.ConstantStepSize(),
                           saveat=P.SaveAt(t1=True)).ys[-1]
        (yT * gy).sum().backward()
        return yT.detach(), y.grad, torch.cat([q.grad.reshape(-1) for q in params])

    def leg(pc):
        for _ in range(max(warmup, 1)):
            step(pc)
        torch.cuda.synchronize()
        # contraction time per launch: one eager step with every launch timed
        lib.pegncde_profile_enable(1)
        eager = step(pc)
        torch.cuda.synchronize()
        prof = {}
        for d, nm in ((0, "fwd"), (1, "bwd")):
            a, t_, ms, by, fl = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
            lib.pegncde_profile_read(d, a, t_, ms, by, fl)
            prof[nm] = dict(us_per_launch=1e3 * ms.value / max(t_.value, 1), hbm_bytes_per_launch=by.value, flops_per_launch=fl.value,
                            launches=t_.value)
        lib.pegncde_profile_enable(0)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step(pc)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.cuda.graph(graph):
            out = step(pc)
        graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
        ms_step = e0.elapsed_time(e1) / steps
        res = dict(steps_per_s=B * S / (ms_step * 1e-3), ms_per_step=ms_step, contraction=prof)
        del graph
        return res, tuple(x.clone() for x in eager)

    out = dict(workload=name, n=n, h=h, L=L, T=T, B=B, solver_steps=S, nnz=sparse.nnz, nnz_per_row=sparse.nnz / (B * n),
               sparse_gather_bytes_per_launch=2.0 * sparse.nnz * h * 4)
    s_res, s_out = leg(sparse)
    out["sparse"] = s_res
    if edge_grads:
        sg = sparse.with_x(None)
        sg.adj_packed = sparse.coef.detach().clone().requires_grad_(True)
        g_res, g_out = leg(sg)
        g_res["kernels"] = kernel_times(step, sg)
        g_res["g_adj_finite"] = bool(torch.isfinite(sg.adj_packed.grad).all())
        out["sparse_edge_grads"] = g_res
        out["edge_grads_throughput_ratio"] = g_res["steps_per_s"] / s_res["steps_per_s"]
        out["edge_grads_outputs_bit_identical"] = bool(torch.equal(g_out[0], s_out[0]) and torch.equal(g_out[1], s_out[1]))
    if dense is not None:
        d_res, d_out = leg(dense)
        out["dense"] = d_res
        out["dense_plane_bytes"] = dense.adj_coef.numel() * 4
        out["max_rel_diff"] = dict(yT=rel(s_out[0], d_out[0]), g_y0=rel(s_out[1], d_out[1]), g_params=rel(s_out[2], d_out[2]))
        out["sparse_speedup"] = s_res["steps_per_s"] / d_res["steps_per_s"]
    else:
        out["dense"] = None
        out["dense_plane_bytes_needed"] = B * (T - 1) * 16.0 * ((n + 31) // 32 * 32) ** 2
        out["finite"] = bool(all(torch.isfinite(x).all() for x in s_out))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--edge-grads", action="store_true", help="also time the solve with the cotangent of the sparse coefficients")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    dev = torch.device("cuda:0")
    info = gpu_info()
    rows = [measure(nm, WORKLOADS[nm], args.steps, args.warmup, dev, args.edge_grads) for nm in args.workloads.split(",")]
    info_end = gpu_info()
    both = [r for r in rows if r["dense"] is not None]
    wins = [r["n"] for r in both if r["sparse_speedup"] > 1.0]
    loses = [r["n"] for r in both if r["sparse_speedup"] <= 1.0]
    if wins and loses:
        cross = f"the sparse control is slower at n = {loses} and faster at n = {wins}: the crossover lies between"
    elif wins:
        cross = f"the sparse control is faster at every measured n ({wins})"
    else:
        cross = f"the sparse control is slower at every measured n ({loses})"
    print(json.dumps(dict(gpu=info, sm_mhz_after=info_end.get("sm_mhz"), steps=args.steps, warmup=args.warmup, workloads=rows,
                          crossover=cross)))


if __name__ == "__main__":
    main()
