#!/usr/bin/env python
"""Benchmark of the FSRNet train step (BASELINE.json metric: FSRNet train imgs/sec @16->128).

  python bench.py [--gpus N --steps K --warmup W]            our arm: native sm_100a hot path
  python bench.py --impl reference [...]                     the reference algorithm on the host CPU cores (oracle port)
  python bench.py --dump-outputs DIR [...]                   also write what the last timed step computed to DIR/*.npy

A "step" is one pass of the hot path over one synthetic batch of `--batch` faces per GPU (config 2 of BASELINE.json:
bf16, batch 128, 16x16 -> 128x128 with parsing-map and landmark priors): bicubic 8x upsample of the uint8 LR faces,
coarse SR net, encoder, hourglass prior estimator, decoder, pixel + prior losses, full backward, bucketed NCCL
gradient all-reduce (N > 1) and the RMSprop update.  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_IMG_TRAIN = 149.9e9      # SURVEY.md 8(d): 3 x 24.983 GMAC x 2
METRIC = "fsrnet_train_images_per_sec"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons while the timed region runs: ONE nvidia-smi process in loop mode
    (-lms 100) streamed line by line (a query per sample costs ~0.4 s of start-up each and yields 1-2 samples)."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None
        self.t_start = float("inf")      # samples before the timed region starts are discarded

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.strip().split(",")]
                if len(f) >= 6 and time.perf_counter() >= self.t_start:
                    self.rows.append(f)
                if self.stop_flag:
                    break
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        self.join(timeout=3)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def cpu_reference_step_rate(steps, warmup, batch=4, size=128):
    """The reference's FSRNet train step on the host cores (fp32, config 1 of BASELINE.json): forward + losses + backward
    + RMSprop.  With oracle/_ref (the reference's own modules, byte-compiled by oracle/build_ref.py in the build container)
    this runs THE REFERENCE - model/FSRnet.py, loss/loss.py, torch.optim.RMSprop as FSR_main.py:185,231-251 - and reports
    kind "reference"; without it, the oracle port (kind "port").  Returns (images/s, cores, s/step, kind, what)."""
    import torch
    from oracle import build_ref as BR
    from oracle import fsrnet_oracle as FO
    from oracle import ref_loader as RL
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    x, hr, lbl, hm = FO.synthetic_batch(batch, size)
    if BR.available():
        F, Ls = BR.load("FSRnet"), BR.load("loss")
        torch.manual_seed(1234)
        net = F.OverallNetwork()
        net.apply(RL.reference_weights_init)
        net.train()
        mse, lmk, ce = Ls.MSELossFunc(), Ls.MSELoss_Landmark(), Ls.CrossEntropyLoss2d()
        opt = torch.optim.RMSprop(net.parameters(), lr=1e-3, alpha=0.99, weight_decay=1e-5)
        kind, what = "reference", "the reference's own modules (oracle/_ref: model/FSRnet.py, loss/loss.py) + torch RMSprop"

        def step():
            outs = RL.reference_fsrnet_forward(net, x)
            total = (5. * mse(outs[1], hr) + 5. * mse(outs[0], hr) + lmk(outs[2], hm) + ce(outs[3], lbl)) / (2.0 * batch)
            opt.zero_grad()
            total.backward()
            opt.step()
    else:
        sd = FO.build_fsrnet_state_dict(1234)
        leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        live = [v for k, v in leaves.items() if not FO.fsrnet_dead_param(k)]
        opt = torch.optim.RMSprop(live, lr=1e-3, alpha=0.99, weight_decay=1e-5)
        kind, what = "port", "oracle port of model/FSRnet.py + loss/loss.py + torch RMSprop"

        def step():
            outs = FO.fsrnet_forward(leaves, x)
            total, _ = FO.fsrnet_loss(outs, hr, hm, lbl)
            opt.zero_grad()
            total.backward()
            opt.step()
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return batch * len(times) / sum(times), cores, sum(times) / len(times), kind, what


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # every step is batch 4 (about 1-3 s of CPU work)
    value, cores, sec, kind, what = cpu_reference_step_rate(args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "FSRNet train step 16->128 (128x128 input), reference algorithm on host CPU",
                       "sample": "batch 4 per step (config 1 of BASELINE.json)"},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": kind,
                             "sample": "%s, batch 4 x 128x128 per step, fp32" % what},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# dram__bytes_read.sum + dram__bytes_write.sum of one rowconv_pair_kernel launch over 128 images from the committed
# `ncu --set full` capture of this round (profiles/r2_rowconv_pair_final_ncu.txt): 273.3 MB + 224.7 MB (algorithmic: 268.4 MB in
# + 268.4 MB out; part of the output is still dirty in the 126 MB L2 when the kernel ends).  A counter cannot be read
# inside an un-profiled run, so the figure is labelled with its source (`traffic_source`).
ROWCONV_TRAFFIC_BYTES_PER_IMAGE = (273.30e6 + 224.68e6) / 128
ROWCONV_TRAFFIC_SOURCE = "ncu --set full capture profiles/r2_rowconv_pair_final_ncu.txt (round 2 final, rowconv_pair_kernel<0>, 128 images)"


def time_matcher(torch, ops, dist, world, rank, probes=10000, gallery=1000000, dim=512, k=5, reps=8):
    """Cosine-similarity identification (BASELINE.json configs[3]): 10 k probes x 1 M-entry 512-d gallery, top-5.
    N > 1: the gallery rows are sharded across the ranks, every rank runs the fused GEMM + top-k on its shard, the per-rank
    (score, index) lists are all-gathered over NCCL and merged (crfr_b200.utils.cosine_identify(sharded=True))."""
    from crfr_b200.utils import utils as U
    g = torch.Generator(device="cuda").manual_seed(11)             # same seed on every rank: identical gallery / probes
    gal = ops.l2norm_bf16(torch.randn(gallery, dim, generator=g, device="cuda"))
    ids = torch.randint(0, gallery, (probes,), generator=g, device="cuda")
    pr = ops.l2norm_bf16(gal[ids].float() + 0.3 * torch.randn(probes, dim, generator=g, device="cuda") / dim ** 0.5)
    lo, hi = U.shard_rows(gallery, world, rank)
    shard = gal[lo:hi].contiguous()
    del gal

    def run():
        return U.cosine_identify(pr, shard, k, normalized=True, index_base=lo, sharded=world > 1)
    for _ in range(3):                   # warm-up (the first call also sizes the cached workspace)
        val, idx = run()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        val, idx = run()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    hit = float((idx[:, 0].long() == ids).float().mean().item())
    return {"queries_per_sec": probes / (ms * 1e-3), "ms": ms, "tflops": 2.0 * probes * gallery * dim / (ms * 1e-3) / 1e12,
            "rank1_hit_rate": hit, "gallery_shards": world,
            "workload": "%d probes x %d x %d gallery, top-%d, bf16%s" % (
                probes, gallery, dim, k, "" if world == 1 else ", gallery sharded over %d GPUs + all-gather + merge" % world)}


def time_kd_step(torch, dist, world, batch=256, reps=3, teacher_kind="resnet34"):
    """Residual-KD training step (BASELINE.json configs[2] / [4]): HR batch -> frozen teacher (eval), LR batch -> student
    and assistant (train), six MSE terms, both backward passes, gradient all-reduce of both networks (N > 1) and the fused
    RMSprop - crfr_b200.trainer.KDTrainer, per-GPU batch 256.  Device-timed, max over ranks."""
    from crfr_b200.model.model_irse import IR_50
    from crfr_b200.model.resnet import ResNet_34
    from crfr_b200.trainer import KDTrainer
    torch.manual_seed(7)
    nets = [ResNet_34().cuda() for _ in range(3)]
    for n in nets:                       # zero-initialised bn2 weights would make every residual branch vanish
        for k, p in n.named_parameters():
            if k.endswith("bn2.weight"):
                p.data.fill_(0.5)
    teacher, student, assistant = nets
    if teacher_kind == "ir50":
        teacher = IR_50([112, 112]).cuda()
    teacher.eval(); student.train(); assistant.train()
    tr = KDTrainer(teacher, student, assistant, lr=1e-4, use_graph=True)
    x_hr = torch.randn(batch, 3, 112, 112, device="cuda")
    x_lr = torch.randn(batch, 3, 112, 112, device="cuda")
    for _ in range(2):                   # warm-up: kernel attributes, allocator pools for the 9 GB workspaces
        tr.step(x_hr, x_lr)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        losses = tr.step(x_hr, x_lr)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    # SURVEY.md 8(d): student + assistant 2 x 21.53 GFLOP, + 14.35 for dL_a/dtheta_S (propagated), + the teacher's forward
    flop = 2 * 21.53e9 + 14.35e9 + (12.59e9 if teacher_kind == "ir50" else 7.175e9)
    return {"images_per_sec": world * batch / (ms * 1e-3), "ms_per_step": ms, "tflops_per_gpu": batch * flop / (ms * 1e-3) / 1e12,
            "student_loss": float(losses[0].item()), "assistant_loss": float(losses[1].item()),
            "workload": "KDTrainer step: %s teacher (eval, HR batch) + ResNet_34 student + assistant (LR batch), batch %d per "
                        "GPU, 112x112, CUDA-graph replay, all-reduce + RMSprop included" % (teacher_kind, batch)}


def time_ir50(torch, batch=256, reps=3):
    """Frozen IR_50 teacher forward (SURVEY.md 8f-1, DISTILLATION/model/model_irse.py), eval mode, 12.59 GFLOP/image."""
    from crfr_b200.model.model_irse import IR_50
    torch.manual_seed(9)
    net = IR_50([112, 112]).cuda().eval()
    x = torch.randn(batch, 3, 112, 112, device="cuda")
    with torch.no_grad():
        for _ in range(2):
            net(x)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            net(x)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return {"images_per_sec": batch / (ms * 1e-3), "ms": ms, "tflops": batch * 12.59e9 / (ms * 1e-3) / 1e12,
            "workload": "IR_50 teacher forward (eval), batch %d, 112x112" % batch}


def time_dominant_kernel(torch, ops, L, chunk):
    """CUDA-event timing of the dominant kernel: the 3x3 64->64 implicit GEMM at 128x128 (87 % of the MACs)."""
    g = torch.Generator(device="cuda").manual_seed(3)
    c, h = 64, 128
    xs = [torch.randn(chunk, h, h, c, generator=g, device="cuda").to(torch.bfloat16) for _ in range(4)]  # > L2 in total
    w = ops.pack_conv_weight(torch.randn(c, c, 3, 3, generator=g, device="cuda") * 0.05)
    for x in xs:
        ops.conv_fwd(x, w, c, c, 3, 1, 1, engine=L.ENGINE_TCGEN05)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    import ctypes as C
    d = ops.conv_desc(xs[0], c, c, 3, 1, 1)
    y = torch.empty((chunk, h, h, c), dtype=torch.bfloat16, device="cuda")
    ws = ops.workspace(L.lib().crfr_conv_workspace_bytes(C.byref(d)))
    reps = 12
    ev0.record()
    for i in range(reps):
        L.call("crfr_conv_fwd", L.ENGINE_TCGEN05, C.byref(d), xs[i % 4].data_ptr(), w.data_ptr(), c, None, y.data_ptr(),
               None, None, 1e-5, ws.data_ptr(), ws.numel(), ops.stream())
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    flops = 2.0 * chunk * h * h * c * c * 9
    return flops / (ms * 1e-3) / 1e12, ms, flops


# dram__bytes_read.sum + dram__bytes_write.sum over 128 images from the committed `ncu --set full` captures: the row-streaming
# dgrad kernel with the fused first pass (profiles/r2_rowconv_pair_final_ncu.txt, variant 1: 1079.1 + 236.2 MB) and the apply
# pass (profiles/r1_norm_stream_ncu_full.txt, kernel unchanged: 538.7 + 235.3 MB); algorithmic: 8 maps of 268.4 MB (the tail of
# each output map is still dirty in L2 when its kernel ends)
NORM_BWD_TRAFFIC_BYTES_PER_IMAGE = (1079.1e6 + 236.2e6 + 538.7e6 + 235.3e6) / 128


def time_norm_bwd(torch, ops, L, chunk):
    """CUDA-event timing of the dominant HBM-bound op of the step: the backward across conv(PReLU(InstanceNorm(y) + res))
    of a residual block (64 x 128 x 128, second gradient summed in) as crfr_conv_dgrad_norm_bwd - the row-streaming dgrad
    kernel with the first pass of the normalisation backward in its epilogue (dout, db, y, res in, dz out: 5 maps) and the
    apply pass (dz, y in, dy out: 3 maps) = 8 maps of chunk x 2 MiB; rotating buffers > L2."""
    g = torch.Generator(device="cuda").manual_seed(5)
    c, h, sets = 64, 128, 3
    mk = lambda: torch.randn(chunk, h, h, c, generator=g, device="cuda").to(torch.bfloat16)
    ys, das, dbs, rs = ([mk() for _ in range(sets)] for _ in range(4))
    gamma, beta, alpha = (torch.rand(c, device="cuda") + 0.5 for _ in range(3))
    wt = ops.pack_conv_weight(torch.randn(c, c, 3, 3, generator=g, device="cuda") * 0.05, for_dgrad=True)
    stats = ops.norm_stats(ys[0])
    run = lambda k: ops.conv_dgrad_norm_bwd(das[k], wt, ys[k], stats, c, c, 3, 1, 1, gamma, beta, alpha, res=rs[k], dx_b=dbs[k],
                                            engine=L.ENGINE_TCGEN05)
    for i in range(2):
        run(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 12
    e0.record()
    for i in range(reps):
        run(i % sets)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    nbytes = 8.0 * chunk * h * h * c * 2
    return nbytes / (ms * 1e-3) / 1e9, ms, nbytes


def verify_dp(torch, dist, world, rank, dev, per_rank=4, size=128):
    """Data-parallel correctness on hardware: the SUM-all-reduced gradient of `world` ranks with `per_rank` images each
    against the single-GPU gradient of the concatenated batch (computed on every rank, so no extra exchange).  FSRNet uses
    InstanceNorm only, so the two are equal up to fp32 summation order."""
    from crfr_b200.model.FSRnet import OverallNetwork, weights_init
    from crfr_b200.trainer import FSRNetTrainer

    class GradOnly(FSRNetTrainer):
        def _optimizer_step(self, lr):
            pass
    g = torch.Generator().manual_seed(2024)
    n = per_rank * world
    x = torch.randn(n, 3, size, size, generator=g).to(dev)
    hr = torch.randn(n, 3, size, size, generator=g).to(dev)
    hm = torch.rand(n, size // 4, size // 4, generator=g).to(dev)
    lbl = torch.randint(0, 11, (n, 1, size // 4, size // 4), generator=g).to(dev)
    out = []
    for dp in (True, False):
        torch.manual_seed(1234)
        net = OverallNetwork()
        net.apply(weights_init)
        # the single-GPU run walks the same images in chunks of `per_rank`: every chunk is then the same native call a rank
        # makes (identical kernels, partitions and roundings), so the comparison isolates the data-parallel plumbing - loss
        # scaling, bucket coverage, all-reduce - from the chaotic bf16 storage noise of differently partitioned forwards
        tr = GradOnly(net.to(dev).train(), chunk=per_rank, world_size=world if dp else 1)
        if not dp:
            tr.dist = None
        sl = slice(rank * per_rank, (rank + 1) * per_rank) if dp else slice(0, n)
        tr.step(x[sl], hr[sl], hm[sl], lbl[sl])
        torch.cuda.synchronize()
        out.append(tr.flat_g.double().clone())
    rel = ((out[0] - out[1]).norm() / out[1].norm()).item()
    cos = float(out[0] @ out[1] / (out[0].norm() * out[1].norm()))
    return {"rel_err_allreduced_vs_single_gpu": rel, "cosine": cos, "images": n, "ranks": world, "pass": bool(rel < 1e-3)}


OUTPUT_SAMPLE = 1 << 18     # elements kept of each forward output: the dump stays under 64 MB (params + grads are ~56 MB)


def dump_outputs(out_dir, trainer, losses, batch):
    """Writes what the last step computed as float32 DIR/<name>.npy, so that two builds can be compared output for output:
    the losses step() returned (total, L_sr, L_coarse, L_lm, L_ce), the flat parameter arena after the RMSprop update and
    the gradient arena it applied, and - when one chunk holds the whole batch (the default), so that the trainer still
    has them - the four forward outputs, each as the same seeded sample of OUTPUT_SAMPLE elements (flat index order)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"losses": losses, "params": trainer.flat_p, "grads": trainer.flat_g}
    if trainer.outs is not None and trainer.outs[0].shape[0] == batch:
        for name, t in zip(("coarse", "sr", "landmark", "parsing"), trainer.outs):
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), min(OUTPUT_SAMPLE, t.numel()), replace=False))
            arrays["out_" + name] = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import crfr_b200
    crfr_b200.build()
    from crfr_b200 import _lib as L, ops
    from crfr_b200.model.FSRnet import OverallNetwork, weights_init
    from crfr_b200.trainer import FSRNetTrainer

    B, S, LR = args.batch, 128, 16
    torch.manual_seed(1234)
    net = OverallNetwork()
    net.apply(weights_init)
    net = net.to(dev).train()
    trainer = FSRNetTrainer(net, lr=1e-3, chunk=args.chunk, lanes=args.lanes, use_graph=bool(args.graph))

    # synthetic data (SURVEY.md 8d), a few distinct batches in pinned host memory
    g = torch.Generator().manual_seed(4321 + rank)
    nb = 2
    host = []
    for _ in range(nb):
        host.append((torch.randint(0, 256, (B, LR, LR, 3), generator=g, dtype=torch.uint8).pin_memory(),
                     torch.randn(B, 3, S, S, generator=g).pin_memory(),
                     torch.rand(B, S // 4, S // 4, generator=g).pin_memory(),
                     torch.randint(0, 11, (B, 1, S // 4, S // 4), generator=g).pin_memory()))
    resident = [tuple(t.to(dev) for t in hb) for hb in host]
    h2d = sum(t.numel() * t.element_size() for t in host[0])

    def step_resident(i):
        lr_u8, hr, hm, lbl = resident[i % nb]
        _, x = ops.bicubic_u8(lr_u8, S, S, want_f32=True)
        return trainer.step(x, hr, hm, lbl)

    def step_e2e(i):
        hb = host[i % nb]
        lr_u8, hr, hm, lbl = (t.to(dev, non_blocking=True) for t in hb)
        _, x = ops.bicubic_u8(lr_u8, S, S, want_f32=True)
        return float(trainer.step(x, hr, hm, lbl)[0].item())        # device -> host read of the loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()            # nvidia-smi comes up during the warm-up; only samples after t_start are kept
        for i in range(warmup):
            fn(i)
        barrier()
        launches0 = L.lib().crfr_launch_count()
        replays0 = trainer.replays
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler:
            sampler.t_start = time.perf_counter()
        e0.record()
        last = None
        for i in range(steps):
            last = fn(warmup + i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        # eager launches are counted by the library; a CUDA-graph replay re-issues the launches counted during its capture
        launches = L.lib().crfr_launch_count() - launches0 + (trainer.replays - replays0) * trainer.graph_launches
        if sampler:
            sampler.stop()
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), launches, (sampler.summary() if sampler else None), last

    ms, launches, clocks, last = timed(step_resident, args.steps, args.warmup)
    loss_val = float(last[0].item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, last, B)
    ms_e2e, _, _, _ = timed(step_e2e, max(2, args.steps // 2), 1)
    value = world * B * args.steps / (ms * 1e-3)
    e2e = world * B * max(2, args.steps // 2) / (ms_e2e * 1e-3)

    extras = {}
    if not args.no_extras:
        # the other BASELINE.json paths, measured in the same run on all ranks (secondary numbers, not the headline metric)
        trainer.ws = None
        trainer._graph, trainer._static = None, None
        torch.cuda.empty_cache()
        extras["matcher"] = time_matcher(torch, ops, dist, world, rank)
        extras["kd_step"] = time_kd_step(torch, dist, world)
        if world == 1:
            extras["kd_step_ir50_teacher"] = time_kd_step(torch, dist, world, teacher_kind="ir50")
            extras["ir50_teacher"] = time_ir50(torch)
    if args.verify and world > 1:
        extras["dp_verify"] = verify_dp(torch, dist, world, rank, dev)
    if rank == 0:
        burst, sustained, hbm, how = measured_peaks()
        k_tflops, k_ms, k_flops = time_dominant_kernel(torch, ops, L, args.chunk)
        line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "FSRNet train step bf16, batch %d per GPU, 16x16 -> 128x128, parsing + landmark "
                                       "priors (BASELINE.json configs[1])" % B, "global_batch": B * world,
                           "chunk": args.chunk, "lanes": args.lanes, "cuda_graph": bool(args.graph), "parallelism": "dp%d" % world,
                           "l2": "inputs + saved activations per chunk (GBs) exceed the 126 MB L2; no explicit flush"},
                "clocks": clocks, "loss": loss_val,
                "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
                "gpu_launches": int(launches),
                "step_tensor_frac": {"achieved_tflops": value / world * FLOP_PER_IMG_TRAIN / 1e12,
                                     "peak_tflops_sustained": sustained,
                                     "frac": value / world * FLOP_PER_IMG_TRAIN / 1e12 / sustained, "peak": how},
                "roofline": {"bound": "tensor", "kernel": "rowconv_pair_kernel (cta_group::2, 3x3 64->64 @128x128 forward, %d "
                                                          "images per launch)" % args.chunk,
                             "achieved": k_tflops, "peak": burst, "unit": "TFLOP/s", "frac": k_tflops / burst,
                             "traffic": ROWCONV_TRAFFIC_BYTES_PER_IMAGE * args.chunk,
                             "traffic_source": ROWCONV_TRAFFIC_SOURCE, "ms_per_launch": k_ms,
                             "flops_per_launch": k_flops, "peak_source": how}}
        n_gbs, n_ms, n_bytes = time_norm_bwd(torch, ops, L, args.chunk)
        line["roofline_hbm"] = {"bound": "hbm", "kernel": "rowconv_pair_kernel<1> (3x3 dgrad + fused first pass of the InstanceNorm "
                                                          "+ PReLU + residual backward) + norm_bwd_apply_stream_kernel, "
                                                          "64 x 128 x 128, %d images" % args.chunk,
                                "achieved": n_gbs, "peak": hbm, "unit": "GB/s", "frac": n_gbs / hbm,
                                "traffic": NORM_BWD_TRAFFIC_BYTES_PER_IMAGE * args.chunk,
                                "traffic_source": "ncu --set full captures profiles/r2_rowconv_pair_final_ncu.txt (variant 1) + "
                                                  "profiles/r1_norm_stream_ncu_full.txt (apply pass, kernel unchanged)",
                                "ms_per_op": n_ms, "bytes_per_op": n_bytes, "peak_source": how}
        line.update(extras)
        if not args.no_cpu_baseline:
            v, cores, sec, kind, what = cpu_reference_step_rate(3, 1)
            line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": cores, "kind": kind,
                                    "sample": "%s: 3 timed steps of batch 4 x 128x128 fp32 (%.2f s/step)" % (what, sec)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--chunk", type=int, default=128, help="images per native call")
    ap.add_argument("--lanes", type=int, default=1, help="concurrent chunk pipelines (streams) per GPU")
    ap.add_argument("--graph", type=int, default=1, help="1: replay the step from a captured CUDA graph (default), 0: eager")
    ap.add_argument("--verify", action="store_true", help="N > 1: check the all-reduced gradient against the single-GPU "
                                                           "gradient of the concatenated batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the matcher / KD-step secondary measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the losses, parameters, gradients and "
                                                          "a fixed sample of the forward outputs of the last step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the native path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
