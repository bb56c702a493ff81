"""Cost of the identity term in the FSRNet training step (FSRNetTrainer(identity_net=...), crfr_fsrnet_id_train_step).

Usage: python tools/bench_fsrnet_identity.py [--batch 128] [--chunk 128] [--iters 20] [--warmup 3]

At bench.py's configuration (batch 128, one chunk, CUDA graph) it times FSRNetTrainer.step without the identity term,
with an IR_50 teacher and with an IR_SE_50 teacher, alternating the three step by step in one process (one shared
workspace, so that the three fit the card at once), with CUDA events around each step after the warm-up steps.  Then the
module-path composition at the same batch: OverallNetwork through autograd, the 112 x 112 crop, IR_50.forward_features on
it and on the HR crop, F.mse_loss on the five outputs, .backward() (no optimiser step).  Prints the device name and power
limit, then one JSON line.  Writes nothing.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--chunk", type=int, default=128)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    import crfr_b200
    crfr_b200.build()
    from bench_ir50_grad import gpu_info
    from crfr_b200 import _lib as L
    from crfr_b200.loss import CrossEntropyLoss2d, MSELoss_Landmark, MSELossFunc
    from crfr_b200.model import model_irse as IR
    from crfr_b200.model.FSRnet import OverallNetwork, weights_init
    from crfr_b200.trainer import FSRNetTrainer

    B, S = args.batch, 128
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(7)
    x = torch.rand(B, 3, S, S, device=dev, generator=g) * 2 - 1
    hr = torch.rand(B, 3, S, S, device=dev, generator=g) * 2 - 1
    hm = torch.rand(B, S // 4, S // 4, device=dev, generator=g)
    lbl = torch.randint(0, 11, (B, 1, S // 4, S // 4), device=dev, generator=g)

    def fsr():
        torch.manual_seed(1234)
        net = OverallNetwork()
        net.apply(weights_init)
        return net.to(dev).train()

    teachers = {"IR_50": IR.IR_50([112, 112]).to(dev).eval(), "IR_SE_50": IR.IR_SE_50([112, 112]).to(dev).eval()}
    configs = [("off", None), ("IR_50", teachers["IR_50"]), ("IR_SE_50", teachers["IR_SE_50"])]
    trainers = {name: FSRNetTrainer(fsr(), lr=1e-4, chunk=args.chunk, use_graph=True, identity_net=t)
                for name, t in configs}
    c = min(args.chunk, B)
    need = max(tr._ws_need(c, S) for tr in trainers.values())
    shared = torch.empty(need, dtype=torch.uint8, device=dev)
    for tr in trainers.values():
        tr.ws = shared               # steps run one after the other on one stream: one arena serves all three
    times = {name: [] for name, _ in configs}
    for it in range(args.warmup + args.iters):
        for name, _ in configs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            trainers[name].step(x, hr, hm, lbl)
            e1.record()
            torch.cuda.synchronize()
            if it >= args.warmup:
                times[name].append(e0.elapsed_time(e1))
    launches = {name: trainers[name].graph_launches for name, _ in configs}
    del trainers, shared
    torch.cuda.empty_cache()

    # module path: autograd through the drop-in modules, the composition of tests/test_ir50_grad_gpu.py at batch B
    net, t50 = fsr(), teachers["IR_50"]
    mse, lmk, ce = MSELossFunc(), MSELoss_Landmark(), CrossEntropyLoss2d()
    hr_c = hr[:, :, 8:120, 8:120].contiguous()

    def module_step():
        net.zero_grad(set_to_none=True)
        outs = net(x)
        loss = (5. * mse(outs[1], hr) + 5. * mse(outs[0], hr) + lmk(outs[2], hm) + ce(outs[3], lbl)) / (2.0 * B)
        with torch.no_grad():
            f_hr = t50.forward_features(hr_c)
        f_sr = t50.forward_features(outs[1][:, :, 8:120, 8:120])
        (loss + sum(F.mse_loss(a, b) for a, b in zip(f_sr, f_hr))).backward()

    mod = []
    for it in range(args.warmup + args.iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        module_step()
        e1.record()
        torch.cuda.synchronize()
        if it >= args.warmup:
            mod.append(e0.elapsed_time(e1))

    name, power = gpu_info()
    med = {k: statistics.median(v) for k, v in times.items()}
    med["module_IR_50"] = statistics.median(mod)
    print("device: %s, power limit: %s" % (name, power))
    for k, v in times.items():
        print("%-9s median %.2f ms  mean %.2f  min %.2f  max %.2f  (+%.2f ms on the plain step)  graph launches %d"
              % (k, med[k], statistics.mean(v), min(v), max(v), med[k] - med["off"], launches[k]))
    print("module path, IR_50: median %.2f ms  mean %.2f  min %.2f" % (med["module_IR_50"], statistics.mean(mod), min(mod)))
    print(json.dumps({"device": name, "power_limit": power, "batch": B, "chunk": c, "iters": args.iters,
                      "median_ms": med, "graph_launches": launches, "library": os.path.basename(L.LIB_PATH)}))


if __name__ == "__main__":
    main()
