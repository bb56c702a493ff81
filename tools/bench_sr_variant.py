"""Convolution shape classes of the SUPER_RESOLUTION FSRNet variant: CUDA-core direct kernels against the tensor-core paths,
and SRNetwork forward + backward with and without them.

Usage: python tools/bench_sr_variant.py [--batch 32] [--iters 20] [--warmup 3] [--skip-layers] [--skip-net]
       python tools/bench_sr_variant.py --profile      (its own run: the kernels of one shipped forward + backward)

1. Every convolution shape of the variant at a 128 x 128 input, at --batch: forward, dgrad and wgrad on ENGINE_DIRECT and
   on ENGINE_AUTO (the tensor-core paths), CUDA events around 10 launches after 3 warm-up launches.  The inputs rotate
   over as many copies as exceed 256 MB, twice the 126 MB L2, so the operands come from HBM.  FLOP/s are 2 x the
   algorithm's MACs over the measured time.
2. SRNetwork forward + backward at 128 x 128 (loss = sum of the four outputs times fixed random gradients), two arms
   alternating iteration by iteration, --iters timed after --warmup, medians:
     shipped - crfr_b200.functional as it is;
     old     - crfr_b200.functional.conv2d / conv_transpose2d pinned to ENGINE_DIRECT for the shapes that the tensor-core
               paths of this change cover (3x3 / 7x7 padding 0, 1x1 stride 1, 3x3 stride-2 transposed): the routing before
               them, in the same process.  The other layers (3x3 padding 1) stay on ENGINE_AUTO in both arms.
3. --profile: torch.profiler over one shipped forward + backward after a warm-up; every kernel with its count and total
   time, and the CUDA-core convolution kernels (gather_down_kernel, gather_up_kernel, wgrad_kernel) with the layer
   shapes that still call them.
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


def is_new_class(cin, cout, k, stride, pad, transposed):
    """The shapes whose tensor-core paths this benchmark measures (the rest were on the tensor cores before)."""
    if transposed:
        return k == 3 and stride == 2
    return (k == 1 and stride == 1) or (pad == 0 and k in (3, 7))


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


def pin_old_routing(Fn, L):
    """crfr_b200.functional.conv2d / conv_transpose2d with the new shape classes pinned to ENGINE_DIRECT."""
    conv2d, convT = Fn.conv2d, Fn.conv_transpose2d

    def conv2d_old(x, weight, bias=None, stride=1, pad=0, engine=L.ENGINE_AUTO):
        cout, cin, k = weight.shape[0], weight.shape[1], weight.shape[2]
        if is_new_class(cin, cout, k, stride, pad, False):
            engine = L.ENGINE_DIRECT
        return conv2d(x, weight, bias, stride, pad, engine)

    def convT_old(x, weight, stride, pad, out_pad, engine=L.ENGINE_AUTO):
        return convT(x, weight, stride, pad, out_pad, L.ENGINE_DIRECT)

    return (conv2d, convT), (conv2d_old, convT_old)


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
    from crfr_b200 import functional as Fn
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
    x = torch.randn(B, 3, S, S, device=dev, generator=g)
    grads = None

    def step():
        nonlocal grads
        net.zero_grad(set_to_none=True)
        outs = net(x)
        if grads is None:
            grads = [torch.randn(o.shape, device=dev, generator=g) for o in outs]
        torch.autograd.backward(outs, grads)

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        step()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
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
        # the layers that still reach the CUDA-core kernels: the 13- and 68-channel 1x1 prior heads, the 3x3 stem's dgrad
        direct_us = sum(t for _, t in direct.values())
        print("CUDA-core convolution kernels: %s, %.1f us of %.1f us (%.2f %%)" % (
            {n[:60]: c for n, (c, _) in direct.items()}, direct_us, total, 100.0 * direct_us / max(total, 1e-9)))
        result["profile"] = {"total_kernel_us": total, "direct_conv_us": direct_us,
                             "direct_conv_kernels": {n[:80]: c for n, (c, _) in direct.items()}}
        print(json.dumps(result))
        return

    if not args.skip_layers:
        result["layers"] = time_layers(args.batch, gpu)
    if not args.skip_net:
        (c2, ct), (c2_old, ct_old) = pin_old_routing(Fn, L)
        arms = {"shipped": (c2, ct), "old_routing": (c2_old, ct_old)}
        times = {a: [] for a in arms}
        try:
            for it in range(args.warmup + args.iters):
                for arm, (a, b) in arms.items():
                    Fn.conv2d, Fn.conv_transpose2d = a, b
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    step()
                    e1.record()
                    torch.cuda.synchronize()
                    if it >= args.warmup:
                        times[arm].append(e0.elapsed_time(e1))
        finally:
            Fn.conv2d, Fn.conv_transpose2d = c2, ct
        med = {a: statistics.median(v) for a, v in times.items()}
        for a, v in times.items():
            print("SRNetwork fwd+bwd batch %d, %-11s median %.2f ms  min %.2f  max %.2f" % (B, a, med[a], min(v), max(v)))
        print("speed-up of the shipped routing: %.2fx" % (med["old_routing"] / med["shipped"]))
        result["net_median_ms"] = med
    print(json.dumps(result))


if __name__ == "__main__":
    main()
