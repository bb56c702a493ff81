"""Convolution shape classes of the SUPER_RESOLUTION FSRNet variant: CUDA-core direct kernels against the tensor-core paths,
and SRNetwork forward + backward as the network program against the op-by-op composition.

Usage: python tools/bench_sr_variant.py [--batch 32] [--iters 20] [--warmup 3] [--skip-layers] [--skip-net]
       python tools/bench_sr_variant.py --profile      (its own run: the kernels of one shipped forward + backward)

1. Every convolution shape of the variant at a 128 x 128 input, at --batch: forward, dgrad and wgrad on ENGINE_DIRECT and
   on ENGINE_AUTO (the tensor-core paths), CUDA events around 10 launches after 3 warm-up launches.  The inputs rotate
   over as many copies as exceed 256 MB, twice the 126 MB L2, so the operands come from HBM.  FLOP/s are 2 x the
   algorithm's MACs over the measured time.
2. SRNetwork forward + backward at 128 x 128 (loss = sum of the four outputs times fixed random gradients), three arms
   alternating step by step, --iters timed after --warmup, CUDA events, medians.  The inputs rotate over as many batches
   as exceed 256 MB:
     program  - the module (crfr_srnet_forward / crfr_srnet_backward, one autograd node), eagerly;
     graph    - the same two calls captured once into a CUDA graph over a fixed workspace, replayed;
     composed - the op-by-op composition the module ran before (oracle/sr_composed.py).
   Also launches per forward + backward (crfr_launch_count) for each arm and the workspace bytes per image.
3. --profile: torch.profiler over one program forward + backward after a warm-up; every kernel with its count and total
   time, the CUDA-core convolution kernels (gather_down_kernel, gather_up_kernel, wgrad_kernel), and the prior heads'
   own kernels (sr_heads_*) and their GEMM (the one tc_gemm launch of 64 -> 128 channels, timed with CUDA events).
Prints the device name and power limit, then one JSON line.  Writes nothing.
"""
import argparse
import json
import os
import re
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

# (class, cin, cout, k, stride, pad, transposed, input size) at a 128 x 128 network input
SHAPES = [
    ("3x3 s1 p0", 64, 64, 3, 1, 0, False, 130), ("3x3 s1 p0", 128, 128, 3, 1, 0, False, 130),
    ("3x3 s1 p0", 128, 128, 3, 1, 0, False, 66), ("3x3 s1 p0", 256, 256, 3, 1, 0, False, 66),
    ("3x3 s1 p0", 256, 256, 3, 1, 0, False, 34), ("3x3 s1 p0", 512, 512, 3, 1, 0, False, 34),
    ("3x3 s2 p0", 64, 128, 3, 2, 0, False, 130), ("3x3 s2 p0", 128, 256, 3, 2, 0, False, 130),
    ("3x3 s2 p0", 128, 256, 3, 2, 0, False, 66), ("3x3 s2 p0", 256, 512, 3, 2, 0, False, 66),
    ("convT 3x3 s2", 512, 256, 3, 2, 1, True, 32), ("convT 3x3 s2", 256, 128, 3, 2, 1, True, 32),
    ("convT 3x3 s2", 256, 128, 3, 2, 1, True, 64), ("convT 3x3 s2", 128, 64, 3, 2, 1, True, 64),
    ("1x1 s1", 64, 64, 1, 1, 0, False, 128), ("1x1 s1", 64, 64, 1, 1, 0, False, 64), ("1x1 s1", 64, 64, 1, 1, 0, False, 32),
    ("1x1 s1", 64, 64, 1, 1, 0, False, 16), ("1x1 s1", 64, 64, 1, 1, 0, False, 8),
    ("7x7 s1 p0 stem", 3, 64, 7, 1, 0, False, 134), ("3x3 s1 p0 stem", 3, 64, 3, 1, 0, False, 130),
    ("3x3 s1 p0 head", 64, 3, 3, 1, 0, False, 130), ("3x3 s1 p0 head", 128, 3, 3, 1, 0, False, 130),
]


def out_size(k, stride, pad, transposed, size):
    return (size - 1) * stride - 2 * pad + k + 1 if transposed else (size + 2 * pad - k) // stride + 1


def macs(batch, cin, cout, k, stride, pad, transposed, size):
    o = out_size(k, stride, pad, transposed, size)
    return batch * (size * size if transposed else o * o) * cin * cout * k * k


def time_layers(batch, gpu):
    import torch
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    dev = torch.device("cuda", 0)
    rows = []
    for cls, cin, cout, k, stride, pad, tr, size in SHAPES:
        o = out_size(k, stride, pad, tr, size)
        in_ld, out_ld = (4 if cin < 8 else cin), (4 if cout < 8 else cout)
        per = batch * (size * size * in_ld + o * o * out_ld) * 2
        copies = max(2, min(16, -(-(256 << 20) // per)))
        g = torch.Generator(device=dev).manual_seed(1)
        xs = [torch.randn(batch, size, size, in_ld, device=dev, generator=g).bfloat16() for _ in range(copies)]
        dys = [torch.randn(batch, o, o, out_ld, device=dev, generator=g).bfloat16() for _ in range(copies)]
        w = torch.randn((cin, cout, k, k) if tr else (cout, cin, k, k), device=dev, generator=g) / (cin * k * k) ** 0.5
        wp = ops.pack_conv_weight(w, transposed=tr, s_pad=in_ld if cin < 8 else None)
        wt = ops.pack_conv_weight(w, for_dgrad=True, transposed=tr)
        ops_ = {
            "fwd": lambda e, i: ops.conv_fwd(xs[i], wp, cin, cout, k, stride, pad, engine=e, transposed=tr, out_hw=(o, o),
                                             out_ld=out_ld),
            "dgrad": lambda e, i: ops.conv_dgrad(dys[i], wt, tuple(xs[i].shape), cin, cout, k, stride, pad, engine=e,
                                                 transposed=tr),
            "wgrad": lambda e, i: ops.conv_wgrad(xs[i], dys[i], cin, cout, k, stride, pad, engine=e, transposed=tr),
        }
        flop = 2.0 * macs(batch, cin, cout, k, stride, pad, tr, size)
        row = {"class": cls, "shape": "%d->%d @%d%s" % (cin, cout, size, " T" if tr else ""), "gflop": flop / 1e9}
        for op, fn in ops_.items():
            for arm, eng in (("direct", L.ENGINE_DIRECT), ("tc", L.ENGINE_AUTO)):
                for i in range(3):
                    fn(eng, i % copies)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(10):
                    fn(eng, i % copies)
                e1.record()
                torch.cuda.synchronize()
                us = e0.elapsed_time(e1) * 100.0          # ms / 10 launches -> us per launch
                row["%s_%s_us" % (op, arm)] = us
                row["%s_%s_tflops" % (op, arm)] = flop / us / 1e6
        rows.append(row)
        print("%-15s %-14s" % (cls, row["shape"]) + "".join(
            "  %s %8.1f/%8.1f us (%6.1f/%6.1f TFLOP/s)" % (op, row[op + "_direct_us"], row[op + "_tc_us"],
                                                          row[op + "_direct_tflops"], row[op + "_tc_tflops"])
            for op in ("fwd", "dgrad", "wgrad")), flush=True)
        del xs, dys
        torch.cuda.empty_cache()
    return rows


def graph_step(net, xs, grads, L):
    """crfr_srnet_forward + crfr_srnet_backward on a fixed workspace, captured into one CUDA graph; returns replay(i)
    for input batch i (the batches are copied into the captured input buffer first)."""
    import ctypes as C
    import torch
    from crfr_b200 import ops
    b, _, h, w = xs[0].shape
    sd = dict(net.named_parameters())
    params = [sd[k].detach() for k in net.state_dict().keys()]
    pgrads = [torch.zeros_like(p) for p in params]
    table = lambda ts: (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    ws = torch.empty(L.lib().crfr_srnet_workspace_bytes(L.SRNET_NETWORK, b, h, w, 1), dtype=torch.uint8, device=xs[0].device)
    x = xs[0].clone()
    outs = [torch.empty(g.shape, device=x.device) for g in grads]
    io = L.SrnetIO()
    io.section, io.batch, io.h, io.w, io.x = L.SRNET_NETWORK, b, h, w, x.data_ptr()
    for i, o in enumerate(outs):
        io.out[i] = o.data_ptr()
    pt, gt, dt = table(params), table(pgrads), table(grads)

    def calls():
        for t in pgrads:
            t.zero_()
        L.call("crfr_srnet_forward", L.ENGINE_AUTO, pt, C.byref(io), 1, ws.data_ptr(), ws.numel(), ops.stream())
        L.call("crfr_srnet_backward", L.ENGINE_AUTO, pt, gt, C.byref(io), dt, None, ws.data_ptr(), ws.numel(), ops.stream())

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        calls()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        calls()

    def replay(i):
        x.copy_(xs[i])
        graph.replay()
    return replay, ws.numel()


def time_heads_gemm(B, S, dev):
    """The prior heads' 1x1 GEMMs at the program's shapes (recipe 6 stands in: 64 -> 128 forward, 128 -> 64 dgrad,
    X^T dY wgrad), CUDA events around 10 launches after 3 warm-up launches."""
    import torch
    from crfr_b200 import ops
    x = torch.randn(B, S, S, 64, device=dev).bfloat16()
    dy = torch.randn(B, S, S, 128, device=dev).bfloat16()
    w = torch.randn(128, 64, 1, 1, device=dev) / 8
    wp, wt = ops.pack_conv_weight(w), ops.pack_conv_weight(w, for_dgrad=True)
    fns = [lambda: ops.conv_fwd(x, wp, 64, 128, 1, 1, 0), lambda: ops.conv_dgrad(dy, wt, tuple(x.shape), 64, 128, 1, 1, 0),
           lambda: ops.conv_wgrad(x, dy, 64, 128, 1, 1, 0)]
    out = []
    for fn in fns:
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) * 100.0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--skip-layers", action="store_true")
    ap.add_argument("--skip-net", action="store_true")
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    import torch
    import crfr_b200
    crfr_b200.build()
    from bench_ir50_grad import gpu_info
    from crfr_b200 import _lib as L
    from crfr_b200.SUPER_RESOLUTION.model.FSRnet import SRNetwork
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    gpu = gpu_info()
    print("device: %s, power limit: %s" % gpu, flush=True)
    dev = torch.device("cuda", 0)
    result = {"device": gpu[0], "power_limit": gpu[1], "batch": args.batch}

    torch.manual_seed(5)
    net = SRNetwork().to(dev).train() if (args.profile or not args.skip_net) else None
    B, S = args.batch, 128
    g = torch.Generator(device=dev).manual_seed(11)
    copies = max(2, -(-(256 << 20) // (B * 3 * S * S * 4)))
    xs = [torch.randn(B, 3, S, S, device=dev, generator=g) for _ in range(copies)]
    grads = [torch.randn(s, device=dev, generator=g) for s in [(B, 3, S, S), (B, 3, S, S), (B, 68, S, S), (B, 13, S, S)]]

    def step(i, fwd=None):
        net.zero_grad(set_to_none=True)
        outs = (fwd or net)(xs[i % copies])
        torch.autograd.backward(outs, grads)

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        step(0)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(1)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA":
                c, t = kern.get(ev.name, (0, 0.0))
                kern[ev.name] = (c + 1, t + ev.device_time)
        total = sum(t for _, t in kern.values())
        print("kernels of one SRNetwork forward + backward (batch %d, 128 x 128), by total time:" % B)
        for name, (c, t) in sorted(kern.items(), key=lambda kv: -kv[1][1]):
            print("  %9.1f us %5d x  %s" % (t, c, name[:150]))
        cuda_core = re.compile(r"(^|[^a-z_])(gather_down_kernel|gather_up_kernel|wgrad_kernel)\b")
        direct = {n: v for n, v in kern.items() if cuda_core.search(n)}
        direct_us = sum(t for _, t in direct.values())
        heads = {n: v for n, v in kern.items() if "sr_heads" in n}
        heads_us = sum(t for _, t in heads.values())
        print("CUDA-core convolution kernels: %s, %.1f us of %.1f us (%.2f %%)" % (
            {n[:60]: c for n, (c, _) in direct.items()}, direct_us, total, 100.0 * direct_us / max(total, 1e-9)))
        gemm_us = time_heads_gemm(B, S, dev)
        print("prior heads: sr_heads_* kernels %.1f us (%s), 64 -> 128 GEMM forward %.1f us, dgrad %.1f us, wgrad %.1f us"
              % (heads_us, {n[:40]: c for n, (c, _) in heads.items()}, *gemm_us))
        result["profile"] = {"total_kernel_us": total, "direct_conv_us": direct_us,
                             "direct_conv_kernels": {n[:80]: c for n, (c, _) in direct.items()},
                             "heads_kernels_us": heads_us, "heads_gemm_fwd_dgrad_wgrad_us": gemm_us}
        print(json.dumps(result))
        return

    if not args.skip_layers:
        result["layers"] = time_layers(args.batch, gpu)
    if not args.skip_net:
        from oracle import sr_composed as SC
        replay, ws_bytes = graph_step(net, xs, grads, L)
        arms = {"program": lambda i: step(i), "graph": replay, "composed": lambda i: step(i, lambda t: SC.network(net, t))}
        times = {a: [] for a in arms}
        launches = {}
        for it in range(args.warmup + args.iters):
            for arm, fn in arms.items():
                torch.cuda.synchronize()
                n0 = L.lib().crfr_launch_count()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn(it)
                e1.record()
                torch.cuda.synchronize()
                launches[arm] = L.lib().crfr_launch_count() - n0
                if it >= args.warmup:
                    times[arm].append(e0.elapsed_time(e1))
        med = {a: statistics.median(v) for a, v in times.items()}
        for a, v in times.items():
            print("SRNetwork fwd+bwd batch %d, %-8s median %.2f ms  min %.2f  max %.2f  (%d native launches per step)"
                  % (B, a, med[a], min(v), max(v), launches[a]))
        print("program speed-up over the composed path: %.2fx eager, %.2fx graph"
              % (med["composed"] / med["program"], med["composed"] / med["graph"]))
        print("workspace: %.1f MB per image (training arena %.2f GB at batch %d)" % (ws_bytes / B / 2 ** 20, ws_bytes / 2 ** 30, B))
        result["net_median_ms"] = med
        result["launches_per_step"] = launches
        result["workspace_bytes_per_image"] = ws_bytes / B
    print(json.dumps(result))


if __name__ == "__main__":
    main()
