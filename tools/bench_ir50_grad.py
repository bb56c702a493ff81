"""Throughput of IR_50([112, 112]) forward and forward + input gradient (crfr_ir50_backward) at the KD batch size.

Usage: python tools/bench_ir50_grad.py [--batch 256] [--iters 20] [--warmup 3] [--arch ir50]

--arch ir_se50 | ir101 | ir152 | ir_se101 | ir_se152 times the other IR / IR-SE teachers instead (crfr_irnet_*).

Times, with CUDA events after warm-up and in one process:
  * forward only (no grad: the shared-workspace path) and forward + input gradient (autograd path, all five outputs seeded),
    reported as images/s and GFLOP/s with the FLOPs counted from the layer shapes below;
  * the backward alone, repeated on one saved forward;
  * for the SE variants, the device time of each SE kernel in one forward + backward (torch.profiler, a separate pass) next
    to the bytes it moves.
Prints the device name and power limit, then one JSON line.  Writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


ARCHS = {"ir50": ("IR_50", 50, 0), "ir_se50": ("IR_SE_50", 50, 1), "ir101": ("IR_101", 100, 0),
         "ir152": ("IR_152", 152, 0), "ir_se101": ("IR_SE_101", 100, 1), "ir_se152": ("IR_SE_152", 152, 1)}
UNITS = {50: (3, 4, 14, 3), 100: (3, 13, 30, 3), 152: (3, 8, 36, 3)}


def block_specs(num_layers):
    """(in_channel, depth, stride) of the bottleneck units (DISTILLATION/model/model_irse.py get_blocks)."""
    specs, in_ch = [], 64
    for units, depth in zip(UNITS[num_layers], (64, 128, 256, 512)):
        for u in range(units):
            specs.append((in_ch, depth, 2 if u == 0 else 1))
            in_ch = depth
    return specs


def ir50_flops_per_image(num_layers=50):
    """(forward FLOPs, input-gradient FLOPs) per 112x112 image: 2 * MACs of every convolution and of the linear head.
    The input gradient runs one dgrad of the same size per convolution and per linear layer (element-wise passes and the
    SE units' 1x1 layers on pooled vectors, < 0.01 %, not counted)."""
    macs, s = 112 * 112 * 64 * 3 * 9, 112      # stem 3x3 3 -> 64
    for cin, d, stride in block_specs(num_layers):
        so = s // stride
        macs += s * s * d * cin * 9             # res_layer.1: 3x3 s1 at the input resolution
        macs += so * so * d * d * 9             # res_layer.3: 3x3, stride
        if cin != d:
            macs += so * so * d * cin           # shortcut 1x1 s2
        s = so
    macs += 512 * 7 * 7 * 512                   # output_layer.3
    return 2.0 * macs, 2.0 * macs


def se_kernel_profile(torch, fwd_bwd, B, num_layers):
    """Device time (ms) of each SE kernel over one forward + input gradient, and the bytes it moves (the maps each one
    streams; its small per-image vectors not counted) over that time, GB/s."""
    from torch.profiler import ProfilerActivity, profile
    fwd_bwd()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fwd_bwd()
        torch.cuda.synchronize()
    ms = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            k = kernel_name(e.name)
            if k.startswith("se_") or k == "ir50_bwd_ew_kernel":
                ms[k] = ms.get(k, 0.0) + e.time_range.elapsed_us() / 1e3
    maps, s = 0, 112                            # bf16 elements of all res_layer.3 outputs of the batch
    for cin, d, stride in block_specs(num_layers):
        s //= stride
        maps += B * s * s * d
    # apply: y + shortcut in, out; reduce: g + y in; the SE part of the element-wise backward pass: g in, dr out
    traffic = {"se_apply_kernel": 3 * 2 * maps, "se_bwd_reduce_kernel": 2 * 2 * maps}
    return {k: {"ms": round(v, 3), "gb": round(traffic[k] / 1e9, 3) if k in traffic else None,
                "gb_per_s": round(traffic[k] / v / 1e6, 1) if k in traffic else None} for k, v in sorted(ms.items())}


def kernel_name(sig):
    """'void (anonymous namespace)::foo<3>(float const*, ...)' -> 'foo'"""
    return sig.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0].split("<")[0].strip()


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, power = [v.strip() for v in out[0].split(",")]
        return name, power
    except Exception as e:   # the numbers are still reported, with the reason the card could not be read
        import torch
        return torch.cuda.get_device_name(), "unknown (%s)" % type(e).__name__


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--arch", choices=sorted(ARCHS), default="ir50")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_ir50_grad: needs a CUDA device")
    from crfr_b200.model import model_irse as M
    from oracle import resnet_oracle as RO

    B = args.batch
    ctor, num_layers, se = ARCHS[args.arch]
    torch.manual_seed(91)
    net = getattr(M, ctor)([112, 112])
    if args.arch == "ir50":
        net.load_state_dict(RO.randomize_bn_everywhere(RO.build_ir50_state_dict(91), 191))
    else:   # seeded construction with non-trivial BatchNorm statistics
        net.load_state_dict(RO.randomize_bn_everywhere(net.state_dict(), 191))
    net = net.cuda().eval()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, 3, 112, 112, generator=g).cuda()
    seeds = [t.cuda() for t in (torch.randn(B, 512, generator=g), torch.randn(B, 64, 56, 56, generator=g),
                                torch.randn(B, 128, 28, 28, generator=g), torch.randn(B, 256, 14, 14, generator=g),
                                torch.randn(B, 512, 7, 7, generator=g))]

    def timed(fn, iters):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    def fwd():
        with torch.no_grad():
            net.forward_features(x)

    xg = x.clone().requires_grad_(True)

    def fwd_bwd():
        outs = net.forward_features(xg)
        torch.autograd.grad(outs, xg, seeds)

    t_fwd = timed(fwd, args.iters)
    t_fb = timed(fwd_bwd, args.iters)
    outs = net.forward_features(xg)
    t_bwd = timed(lambda: torch.autograd.grad(outs, xg, seeds, retain_graph=True), args.iters)
    f_fwd, f_bwd = ir50_flops_per_image(num_layers)
    name, power = gpu_info()
    res = {
        "arch": ctor, "device": name, "power_limit": power, "batch": B, "iters": args.iters,
        "gflop_per_image_fwd": round(f_fwd / 1e9, 3), "gflop_per_image_dgrad": round(f_bwd / 1e9, 3),
        "fwd_ms": round(t_fwd, 3), "fwd_images_per_s": round(B / t_fwd * 1e3, 1),
        "fwd_tflops": round(B * f_fwd / t_fwd / 1e9, 1),
        "fwd_grad_ms": round(t_fb, 3), "fwd_grad_images_per_s": round(B / t_fb * 1e3, 1),
        "fwd_grad_tflops": round(B * (f_fwd + f_bwd) / t_fb / 1e9, 1),
        "bwd_ms": round(t_bwd, 3), "bwd_over_fwd": round(t_bwd / t_fwd, 2),
    }
    if se:
        res["se_kernels"] = se_kernel_profile(torch, fwd_bwd, B, num_layers)
    print("device: %s, power limit: %s" % (name, power))
    print(json.dumps(res))

if __name__ == "__main__":
    main()
