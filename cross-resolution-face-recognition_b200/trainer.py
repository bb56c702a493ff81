"""Data-parallel FSRNet training loop (the replacement for the loop body at FSR_main.py:219-251).

One process per GPU.  Per step and per rank:
  1. (optional) bicubic 8x upsample of the uint8 LR faces on the GPU (bit-exact with PIL, crfr_bicubic_u8);
  2. the batch is walked in chunks of ``chunk`` images: each chunk runs forward + losses + backward in ONE native call
     (crfr_fsrnet_train_step).  InstanceNorm only -> samples are independent, so chunking is exact; it keeps a chunk's
     2 MiB/img activation maps L2-resident between consecutive kernels and bounds the workspace;
  3. gradients accumulate in one flat fp32 arena laid out in state_dict order, so the three all-reduce buckets
     (decoder | prior+encoder | coarse = reverse execution order) are contiguous slices.  During the LAST chunk's
     backward the native program records a CUDA event as each bucket becomes final; the bucket's NCCL all-reduce is
     issued on a side stream behind that event and overlaps the rest of the backward (only collective in the loop);
  4. fused RMSprop on the flat arena (torch.optim.RMSprop semantics, FSR_main.py:185).

Concurrent lanes (``lanes`` > 1, CUDA only): the chunks are dealt to independent pipelines, each with its own CUDA
stream, workspace and gradient arena.  InstanceNorm makes the chunks independent, so lane A's tensor-bound convolution
kernels overlap lane B's HBM-bound normalisation kernels instead of alternating with them on one stream; the lane
arenas are summed per bucket right before the bucket's all-reduce / the optimiser step.

CUDA graph (``use_graph=True``): the native step issues ~1 100 launches (each conv encodes three tensor maps on the
host), i.e. 20-25 ms of host time per 128 images - as long as one lane keeps the GPU busy for longer than that the
host runs ahead and nothing is lost, but several lanes double the launch count and become host-bound.  With
``use_graph`` the forward + loss + backward of all chunks / lanes is captured once per input shape (stream capture
follows the lane streams and the library's internal weight-gradient stream through their fork / join events) and
replayed from static input buffers; only the all-reduce and the optimiser step stay outside the graph.

Loss scaling: FSR_main.py:234 divides by 2*train_batch.  With G = global batch (all ranks) and chunk size c, the
chunk's share of the batch-mean losses is c/G, so each chunk is run with loss_div = 2*G*G/c and gradients are
SUM-reduced across ranks: the result equals the single-GPU gradient of the concatenated batch.

Identity term (``identity_net``, a frozen 112 x 112 IR / IR-SE ``Backbone`` in eval mode): every chunk runs
crfr_fsrnet_id_train_step instead, which adds w_id * sum_k MSE(f(sr)[k], f(hr)[k]) over the selected outputs of
f = identity_net.forward_features on the 112 x 112 centres (SUPER_RESOLUTION/train_FHN.py:255-265).  Each MSE is a mean
over the chunk, run with id_scale = c/G, so the summed chunk gradients, SUM-reduced across ranks, are again those of
the global-batch mean.  The losses then have a sixth entry, the identity term.
"""
import ctypes as C

import torch

from . import _lib as L
from . import ops
from .model import FSRnet as M

# state_dict index ranges of the all-reduce buckets, in the order they become ready during backward
BUCKET_PARAM_RANGES = ((167, 202), (33, 167), (0, 33))


def flat_layout(shapes, align=4):
    """Offsets (in elements) of each tensor in a flat arena, every tensor 16-byte aligned."""
    offs, tot = [], 0
    for s in shapes:
        n = 1
        for d in s:
            n *= d
        offs.append(tot)
        tot += (n + align - 1) // align * align
    return offs, tot


def bucket_slices(offs, total, ranges=BUCKET_PARAM_RANGES):
    """Contiguous [start, end) element ranges of the flat arena for each bucket."""
    out = []
    for lo, hi in ranges:
        out.append((offs[lo], offs[hi] if hi < len(offs) else total))
    return out


def live_ranges(offs, total, dead):
    """Contiguous [start, end) element ranges of the flat arena that hold live (gradient-receiving) parameters."""
    out, start = [], None
    n = len(offs)
    for i in range(n + 1):
        live = i < n and i not in dead
        if live and start is None:
            start = offs[i]
        if not live and start is not None:
            out.append((start, offs[i] if i < n else total))
            start = None
    return out


def chunk_loss_div(global_batch, chunk):
    """loss_div for one chunk so that the summed chunk gradients equal the gradient of FSR_main.py:233-234."""
    return 2.0 * global_batch * global_batch / chunk


class _Lane:
    """One independent chunk pipeline: stream, workspace, gradient arena, loss accumulators, bucket events."""

    def __init__(self, trainer, index):
        dev = trainer.device
        self.index = index
        self.stream = torch.cuda.Stream(device=dev)
        self.flat_g = trainer.flat_g if index == 0 else torch.zeros_like(trainer.flat_g)
        params = trainer.model.ordered_parameters()
        self.grad_views = [self.flat_g[o:o + p.numel()].view(p.shape) for p, o in zip(params, trainer.offs)]
        self.gtable = M._ParamTable(self.grad_views)
        self.losses = torch.zeros((trainer.n_losses,), dtype=torch.float32, device=dev)
        self.loss_acc = torch.zeros((trainer.n_losses,), dtype=torch.float32, device=dev)
        self.events = [torch.cuda.Event() for _ in trainer.buckets]
        for e in self.events:
            e.record()
        self.done = torch.cuda.Event()
        self.ws = None
        self.outs = None


def _identity_tables(net, terms):
    """Checks the identity teacher and the selected outputs -> (parameter table, buffer table, terms bit mask)."""
    from .model import model_irse as IR
    if not isinstance(net, IR.Backbone):
        raise TypeError("identity_net must be an IR / IR-SE Backbone (model_irse), got %s" % type(net).__name__)
    if not net._native:
        raise NotImplementedError("only the 112 x 112 IR / IR_SE backbones have a native network program")
    if net.training:
        raise RuntimeError("identity_net is the frozen teacher: call .eval() first (train-mode Dropout is stochastic and "
                           "has no parity definition)")
    terms = tuple(terms)
    if not terms or any(k not in range(5) for k in terms) or len(set(terms)) != len(terms):
        raise ValueError("id_terms must be distinct indices into (embedding, x1, x2, x3, x4), got %s" % (terms,))
    n_params, n_bn = L.irnet_sizes(*net._variant)
    params = [p.detach() for _, p in net.named_parameters()]
    buffers = [t for _, t in net.named_buffers()]
    return IR._Table(params, n_params), IR._Table(buffers, 3 * n_bn), sum(1 << k for k in terms)


class FSRNetTrainer:
    def __init__(self, model, lr=1e-3, alpha=0.99, eps=1e-8, weight_decay=1e-5, chunk=16, w_pix=5.0,
                 engine=L.ENGINE_AUTO, process_group=None, world_size=None, lanes=1, use_graph=False, identity_net=None,
                 w_id=1.0, id_terms=(0, 1, 2, 3, 4)):
        import torch.distributed as dist
        self.model = model
        self.identity_net, self.w_id = identity_net, float(w_id)
        self._id_tabs = None if identity_net is None else _identity_tables(identity_net, id_terms)
        self.n_losses = 5 if identity_net is None else 6
        self.lr, self.alpha, self.eps, self.wd = lr, alpha, eps, weight_decay
        self.chunk, self.w_pix, self.engine = chunk, w_pix, engine
        self.dist = dist if (dist.is_available() and dist.is_initialized()) else None
        self.pg = process_group
        self.world = world_size if world_size is not None else (self.dist.get_world_size(self.pg) if self.dist else 1)
        params = model.ordered_parameters()
        dev = params[0].device
        self.device = dev
        offs, tot = flat_layout([tuple(p.shape) for p in params])
        self.offs, self.total = offs, tot
        self.flat_p = torch.zeros(tot, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(tot, dtype=torch.float32, device=dev)
        self.flat_sq = torch.zeros(tot, dtype=torch.float32, device=dev)
        self.grad_views = []
        for p, o in zip(params, offs):
            v = self.flat_p[o:o + p.numel()].view(p.shape)
            v.copy_(p.data)
            p.data = v                      # parameters now live in the arena (state_dict / optimisers still work)
            self.grad_views.append(self.flat_g[o:o + p.numel()].view(p.shape))
        self.buckets = bucket_slices(offs, tot)
        self.live_ranges = live_ranges(offs, tot, M._DEAD_PARAMS)
        self.ptable = M._ParamTable([p.data for p in params])
        self.gtable = M._ParamTable(self.grad_views)
        self.losses = torch.zeros((self.n_losses,), dtype=torch.float32, device=dev)
        self.loss_acc = torch.zeros((self.n_losses,), dtype=torch.float32, device=dev)
        self.ws = None
        self.outs = None
        if dev.type == "cuda":
            self.comm_stream = torch.cuda.Stream(device=dev)
            self.events = [torch.cuda.Event() for _ in self.buckets]
            for e in self.events:
                e.record()                  # materialise the cudaEvent_t handles
        else:
            self.comm_stream, self.events = None, []
        self.lanes = [_Lane(self, i) for i in range(lanes)] if (dev.type == "cuda" and lanes > 1) else []
        self._w_cache = {}
        self.use_graph = bool(use_graph) and dev.type == "cuda"
        self._graph, self._graph_key, self._static = None, None, None
        self.graph_launches, self.replays = 0, 0     # launch accounting under graph replay (bench.py gpu_launches)

    def reset_optimizer_state(self):
        """The reference re-creates RMSprop every epoch (FSR_main.py:183-185): the square average restarts."""
        self.flat_sq.zero_()

    # -- one native chunk: overridable so that the CPU (gloo) tests can exercise the host logic without a GPU --
    def _native_chunk(self, x, hr, heatmap, labels, outs, loss_div, events):
        b, s = x.shape[0], x.shape[2]
        need = L.lib().crfr_fsrnet_workspace_bytes(b, s, 1)
        if self.ws is None or self.ws.numel() < need:
            self.ws = torch.empty(need, dtype=torch.uint8, device=x.device)
        io = M._io(x, outs, (hr, heatmap, labels), loss_div=loss_div, w_pix=self.w_pix)
        for i, e in enumerate(events or ()):
            io.bucket_events[i] = e.cuda_event
        L.call("crfr_fsrnet_train_step", self.engine, self.ptable.arr, self.gtable.arr, C.byref(io),
               self.losses.data_ptr(), self.ws.data_ptr(), self.ws.numel(), ops.stream())

    def _ws_need(self, b, s):
        if self.identity_net is None:
            return L.lib().crfr_fsrnet_workspace_bytes(b, s, 1)
        return L.lib().crfr_fsrnet_id_workspace_bytes(*self.identity_net._variant, b, s)

    def _id_call(self, io, gtable, losses, ws, id_scale):
        """crfr_fsrnet_id_train_step of one chunk (io: its crfr_fsrnet_io) into gtable / losses over ws."""
        ptab, btab, mask = self._id_tabs
        idio = L.FsrnetIdIO()
        idio.teacher_layers, idio.teacher_se = self.identity_net._variant
        idio.teacher_params = C.cast(ptab.arr, C.c_void_p)
        idio.teacher_buffers = C.cast(btab.arr, C.c_void_p)
        idio.w_id, idio.terms, idio.id_scale = self.w_id, mask, id_scale
        L.call("crfr_fsrnet_id_train_step", self.engine, self.ptable.arr, gtable.arr, C.byref(io), C.byref(idio),
               losses.data_ptr(), ws.data_ptr(), ws.numel(), ops.stream())

    # -- one native chunk with the identity term (id_scale = chunk / global batch): overridable like _native_chunk --
    def _native_id_chunk(self, x, hr, heatmap, labels, outs, loss_div, id_scale, events):
        b, s = x.shape[0], x.shape[2]
        need = self._ws_need(b, s)
        if self.ws is None or self.ws.numel() < need:
            self.ws = torch.empty(need, dtype=torch.uint8, device=x.device)
        io = M._io(x, outs, (hr, heatmap, labels), loss_div=loss_div, w_pix=self.w_pix)
        for i, e in enumerate(events or ()):
            io.bucket_events[i] = e.cuda_event
        self._id_call(io, self.gtable, self.losses, self.ws, id_scale)

    def _chunk(self, x, hr, heatmap, labels, outs, c, G, events):
        if self.identity_net is None:
            self._native_chunk(x, hr, heatmap, labels, outs, chunk_loss_div(G, c), events)
        else:
            self._native_id_chunk(x, hr, heatmap, labels, outs, chunk_loss_div(G, c), c / G, events)

    def _allreduce_bucket(self, k):
        lo, hi = self.buckets[k]
        return self.dist.all_reduce(self.flat_g[lo:hi], op=self.dist.ReduceOp.SUM, group=self.pg, async_op=True)

    def _loss_weights(self, c, B):
        """total adds up over chunks; the parts are chunk means -> weight by c/B (cached device constants)."""
        key = (c, B)
        if key not in self._w_cache:
            self._w_cache[key] = torch.tensor([1.0] + [c / B] * (self.n_losses - 1), device=self.device)
        return self._w_cache[key]

    def _step_lanes(self, x, hr, heatmap, labels, lr, events_for_dp=True, finish=True):
        """Chunks dealt round-robin to concurrent lanes (see the module docstring)."""
        B = x.shape[0]
        G = B * self.world
        dp = self.dist is not None and self.world > 1 and events_for_dp
        main = torch.cuda.current_stream()
        start = torch.cuda.Event()
        start.record(main)
        starts = list(range(0, B, self.chunk))
        used = self.lanes[:min(len(self.lanes), len(starts))]
        for ln in used:
            ln.stream.wait_event(start)
            with torch.cuda.stream(ln.stream):
                ln.flat_g.zero_()
                ln.loss_acc.zero_()
        for ci, s0 in enumerate(starts):
            s1 = min(B, s0 + self.chunk)
            c = s1 - s0
            ln = used[ci % len(used)]
            last_of_lane = ci + len(used) >= len(starts)
            with torch.cuda.stream(ln.stream):
                if ln.outs is None or ln.outs[0].shape[0] != c or ln.outs[0].shape[2] != x.shape[2]:
                    ln.outs = M.alloc_outputs(x[s0:s1])
                need = self._ws_need(c, x.shape[2])
                if ln.ws is None or ln.ws.numel() < need:
                    ln.ws = torch.empty(need, dtype=torch.uint8, device=x.device)
                io = M._io(x[s0:s1], ln.outs, (hr[s0:s1], heatmap[s0:s1], labels[s0:s1]),
                           loss_div=chunk_loss_div(G, c), w_pix=self.w_pix)
                if dp and last_of_lane:
                    for i, e in enumerate(ln.events):
                        io.bucket_events[i] = e.cuda_event
                if self.identity_net is None:
                    L.call("crfr_fsrnet_train_step", self.engine, self.ptable.arr, ln.gtable.arr, C.byref(io),
                           ln.losses.data_ptr(), ln.ws.data_ptr(), ln.ws.numel(), ops.stream())
                else:
                    self._id_call(io, ln.gtable, ln.losses, ln.ws, c / G)
                ln.loss_acc.add_(ln.losses * self._loss_weights(c, B))
                if last_of_lane:
                    ln.done.record(ln.stream)
        if dp:
            works = []
            with torch.cuda.stream(self.comm_stream):
                for k, (lo, hi) in enumerate(self.buckets):
                    for ln in used:
                        self.comm_stream.wait_event(ln.events[k])
                    for ln in used[1:]:
                        self.flat_g[lo:hi].add_(ln.flat_g[lo:hi])
                    works.append(self._allreduce_bucket(k))
            for wk in works:
                wk.wait()
            for ln in used:
                main.wait_event(ln.done)
        else:
            for ln in used:
                main.wait_event(ln.done)
            for ln in used[1:]:
                self.flat_g.add_(ln.flat_g)
        self.loss_acc.copy_(used[0].loss_acc)
        for ln in used[1:]:
            self.loss_acc.add_(ln.loss_acc)
        if finish:
            self._optimizer_step(self.lr if lr is None else lr)
        return self.loss_acc

    def _compute(self, x, hr, heatmap, labels):
        """forward + losses + backward of every chunk into flat_g / loss_acc; no collective, no optimiser step."""
        if self.lanes and x.shape[0] > self.chunk:
            self._step_lanes(x, hr, heatmap, labels, None, events_for_dp=False, finish=False)
            return
        B = x.shape[0]
        G = B * self.world
        self.flat_g.zero_()
        self.loss_acc.zero_()
        for s0 in range(0, B, self.chunk):
            s1 = min(B, s0 + self.chunk)
            c = s1 - s0
            if self.outs is None or self.outs[0].shape[0] != c or self.outs[0].shape[2] != x.shape[2]:
                self.outs = M.alloc_outputs(x[s0:s1])
            self._chunk(x[s0:s1], hr[s0:s1], heatmap[s0:s1], labels[s0:s1], self.outs, c, G, None)
            self.loss_acc.add_(self.losses * self._loss_weights(c, B))

    def _step_graph(self, x, hr, heatmap, labels, lr):
        key = (tuple(x.shape), tuple(hr.shape), tuple(heatmap.shape), tuple(labels.shape), x.dtype, labels.dtype)
        if self._graph is None or self._graph_key != key:
            self._static = tuple(torch.empty_like(t) for t in (x, hr, heatmap, labels))
            for d, t in zip(self._static, (x, hr, heatmap, labels)):
                d.copy_(t)
            self._compute(*self._static)           # eager warm-up: workspaces, kernel attributes, helper streams
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            n0 = L.lib().crfr_launch_count()
            with torch.cuda.graph(graph):
                self._compute(*self._static)
            self.graph_launches = int(L.lib().crfr_launch_count() - n0)    # kernels of ours inside one replay
            self._graph, self._graph_key = graph, key
        else:
            for d, t in zip(self._static, (x, hr, heatmap, labels)):
                d.copy_(t, non_blocking=True)
        self._graph.replay()
        self.replays += 1
        if self.dist is not None and self.world > 1:
            works = [self._allreduce_bucket(k) for k in range(len(self.buckets))]
            for wk in works:
                wk.wait()
        self._optimizer_step(self.lr if lr is None else lr)
        return self.loss_acc

    def step(self, x, hr, heatmap, labels, lr=None):
        """x [B,3,S,S] fp32 (already upsampled + normalised), hr [B,3,S,S], heatmap [B,S/4,S/4], labels int64
        [B,1,S/4,S/4]; all on this rank's device.  Returns the device tensor (total, L_sr, L_coarse, L_lm, L_ce) of
        this rank's share of the global-batch loss (parts are rank-local batch means); with ``identity_net`` a sixth
        entry, the identity term's rank-local batch mean, whose share is part of the total."""
        if self.identity_net is not None and self.identity_net.training:
            raise RuntimeError("identity_net is the frozen teacher: call .eval() first")
        if x.is_cuda:
            M.check_input(x)
            # the native program reads raw pointers: coerce dtype / contiguity here (slices of a bigger batch are fine)
            x, hr, heatmap = x.contiguous().float(), hr.contiguous().float(), heatmap.contiguous().float()
            labels = labels.contiguous().long()
        if self.use_graph and x.is_cuda:
            return self._step_graph(x, hr, heatmap, labels, lr)
        if self.lanes and x.is_cuda and x.shape[0] > self.chunk:
            return self._step_lanes(x, hr, heatmap, labels, lr)
        B = x.shape[0]
        G = B * self.world
        self.flat_g.zero_()
        self.loss_acc.zero_()
        if self.outs is None or self.outs[0].shape[0] != min(self.chunk, B) or self.outs[0].shape[2] != x.shape[2]:
            self.outs = M.alloc_outputs(x[:min(self.chunk, B)])
        works = []
        starts = list(range(0, B, self.chunk))
        for ci, s0 in enumerate(starts):
            s1 = min(B, s0 + self.chunk)
            c = s1 - s0
            outs = self.outs if c == self.outs[0].shape[0] else M.alloc_outputs(x[s0:s1])
            last = ci == len(starts) - 1
            use_events = last and self.dist is not None and self.world > 1 and self.events
            self._chunk(x[s0:s1], hr[s0:s1], heatmap[s0:s1], labels[s0:s1], outs, c, G,
                        self.events if use_events else None)
            self.loss_acc.add_(self.losses * self._loss_weights(c, B))
            if use_events:
                main = torch.cuda.current_stream()
                with torch.cuda.stream(self.comm_stream):
                    for k, ev in enumerate(self.events):
                        self.comm_stream.wait_event(ev)
                        works.append(self._allreduce_bucket(k))
                for wk in works:
                    wk.wait()               # main stream waits for the collectives
                del main
        if self.dist is not None and self.world > 1 and not works:
            for k in range(len(self.buckets)):
                self._allreduce_bucket(k).wait()
        self._optimizer_step(self.lr if lr is None else lr)
        return self.loss_acc

    def _optimizer_step(self, lr):
        # torch.optim.RMSprop skips parameters whose grad is None: the parameters that never influence the outputs (bn_end,
        # residual_next.*, the encoder's conv_mid, the decoder's instance_norm) must not decay towards zero either, so the
        # fused update runs over the live ranges of the arena only
        for lo, hi in self.live_ranges:
            ops.rmsprop_step(self.flat_p[lo:hi], self.flat_g[lo:hi], self.flat_sq[lo:hi], lr, self.alpha, self.eps, self.wd,
                             gscale=1.0)


class _FlatNet:
    """Parameters, gradients and RMSprop state of one network in flat fp32 arenas (named_parameters order)."""

    def __init__(self, net):
        from .model import resnet as R
        params = net.ordered_parameters()
        dev = params[0].device
        offs, tot = flat_layout([tuple(p.shape) for p in params])
        self.net, self.offs, self.total = net, offs, tot
        self.flat_p = torch.zeros(tot, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(tot, dtype=torch.float32, device=dev)
        self.flat_sq = torch.zeros(tot, dtype=torch.float32, device=dev)
        self.grad_views = []
        for p, o in zip(params, offs):
            v = self.flat_p[o:o + p.numel()].view(p.shape)
            v.copy_(p.data)
            p.data = v
            self.grad_views.append(self.flat_g[o:o + p.numel()].view(p.shape))
        if dev.type == "cuda":
            self.tabs = (R._TableOfPointers([p.data for p in params], L.RESNET34_NPARAMS),
                         R._TableOfPointers(net.ordered_buffers(), 3 * L.RESNET34_NBN),
                         R._TableOfPointers(self.grad_views, L.RESNET34_NPARAMS))


class KDTrainer:
    """Data-parallel residual knowledge-distillation loop (the replacement for distill_main.py:42-74 with the optimisers
    of :222-225), one process per GPU.

    Per step and per rank: ONE native call (crfr_kd_train_step) runs the frozen teacher (ResNet_34 or an IR / IR-SE
    backbone, eval), the student and the assistant (ResNet_34, train: per-replica BatchNorm statistics, as the reference's single-device
    semantics) on this rank's share of the batch, the six MSE terms and both backward passes.  Student and assistant
    gradients live in one flat arena each = one all-reduce bucket each (136 MB fp32): the native call records an event
    when the student's gradients are final, its NCCL all-reduce is issued on a side stream behind that event and
    overlaps the assistant's backward; the assistant's bucket follows at the end.  Gradients are SUM-reduced and scaled
    by 1 / world inside the fused RMSprop (every term is a mean over the rank's batch), so the update equals the
    single-GPU update on the concatenated batch up to the per-replica BatchNorm statistics.
    ``x_hr`` feeds the teacher, ``x_lr`` (default: the same tensor, as distill_main.py:59-61) the student and assistant.
    """

    def __init__(self, teacher, student, assistant, lr=1e-4, alpha=0.99, eps=1e-8, weight_decay=1e-5,
                 assistant_grad_to_student=True, process_group=None, world_size=None, use_graph=False):
        import torch.distributed as dist
        self.teacher, self.student, self.assistant = teacher, student, assistant
        self.lr, self.alpha, self.eps, self.wd = lr, alpha, eps, weight_decay
        self.to_student = assistant_grad_to_student
        self.dist = dist if (dist.is_available() and dist.is_initialized()) else None
        self.pg = process_group
        self.world = world_size if world_size is not None else (self.dist.get_world_size(self.pg) if self.dist else 1)
        self.S, self.A = _FlatNet(student), _FlatNet(assistant)
        dev = self.S.flat_p.device
        self.device = dev
        self.losses = torch.zeros((2,), dtype=torch.float32, device=dev)
        if dev.type == "cuda":
            self.comm_stream = torch.cuda.Stream(device=dev)
            self.events = [torch.cuda.Event(), torch.cuda.Event()]
            for e in self.events:
                e.record()
        else:
            self.comm_stream, self.events = None, []
        # CUDA graph (``use_graph=True``): the ~1 300 launches of the native step are captured once per input shape and
        # replayed from static input buffers (-2.8 ms of launch gaps on a 38 ms step); the all-reduces and the optimiser
        # step stay outside the graph, so under data parallelism the student's all-reduce no longer overlaps the
        # assistant's backward (2 x 136 MB over NVLink after the replay).
        self.use_graph = bool(use_graph) and dev.type == "cuda"
        self._graph, self._graph_key, self._static, self._ws = None, None, None, None
        self.graph_launches, self.replays = 0, 0

    def reset_optimizer_state(self):
        """The reference re-creates both RMSprop optimisers every epoch (distill_main.py:222-225)."""
        self.S.flat_sq.zero_()
        self.A.flat_sq.zero_()

    # overridable so that the CPU (gloo) tests can exercise the host logic without a GPU
    def _native_step(self, x_hr, x_lr, events):
        from .model import resnet as R
        R.kd_native_call(self.teacher, self.student, self.assistant, x_hr, x_lr, self.S.tabs, self.A.tabs, self.losses,
                         self.to_student, events, ws=self._ws)

    def _graph_step(self, x_hr, x_lr):
        """Replay of the captured native step (gradient zeroing included) from static input buffers."""
        key = (tuple(x_hr.shape), x_lr is not None)
        if self._graph is None or self._graph_key != key:
            from .model import resnet as R
            self._static = (torch.empty_like(x_hr), None if x_lr is None else torch.empty_like(x_lr))
            self._static[0].copy_(x_hr)
            if x_lr is not None:
                self._static[1].copy_(x_lr)
            need = R.kd_workspace_bytes(self.teacher, x_hr.shape[0])
            self._ws = torch.empty(need, dtype=torch.uint8, device=x_hr.device)     # private: the graph holds its address
            # eager warm-up (kernel attributes, helper streams) with the BatchNorm buffers restored afterwards, so that the
            # first replayed step is the first running-statistics update
            bufs = [b for n in (self.student, self.assistant) for b in n.ordered_buffers()]
            saved = [b.clone() for b in bufs]
            self._native_step(self._static[0], self._static[1], None)
            for b, v in zip(bufs, saved):
                b.copy_(v)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            n0 = L.lib().crfr_launch_count()
            with torch.cuda.graph(graph):
                self.S.flat_g.zero_()
                self.A.flat_g.zero_()
                self._native_step(self._static[0], self._static[1], None)
            self.graph_launches = int(L.lib().crfr_launch_count() - n0)
            self._graph, self._graph_key = graph, key
        else:
            self._static[0].copy_(x_hr, non_blocking=True)
            if x_lr is not None:
                self._static[1].copy_(x_lr, non_blocking=True)
        self._graph.replay()
        self.replays += 1

    def _optimizer_step(self, lr):
        for f in (self.S, self.A):
            ops.rmsprop_step(f.flat_p, f.flat_g, f.flat_sq, lr, self.alpha, self.eps, self.wd, gscale=1.0 / self.world)

    def step(self, x_hr, x_lr=None, lr=None):
        """One KD step on this rank's batch; returns the device tensor (L_s, L_a) of the rank-local batch."""
        if x_hr.is_cuda:
            from .model import resnet as R
            R.check_kd_nets(self.teacher, self.student, self.assistant)
            x_hr = R.check_kd_input(x_hr, "x_hr")
            x_lr = None if x_lr is None else R.check_kd_input(x_lr, "x_lr")
        dp = self.dist is not None and self.world > 1
        graphed = self.use_graph and x_hr.is_cuda
        if graphed:
            self._graph_step(x_hr, x_lr)
        else:
            self.S.flat_g.zero_()
            self.A.flat_g.zero_()
            self._native_step(x_hr, x_lr, self.events if (dp and self.events) else None)
        if dp:
            works = []
            if self.events and not graphed:
                with torch.cuda.stream(self.comm_stream):
                    for f, ev in zip((self.S, self.A), self.events):
                        self.comm_stream.wait_event(ev)
                        works.append(self.dist.all_reduce(f.flat_g, op=self.dist.ReduceOp.SUM, group=self.pg, async_op=True))
            else:
                works = [self.dist.all_reduce(f.flat_g, op=self.dist.ReduceOp.SUM, group=self.pg, async_op=True)
                         for f in (self.S, self.A)]
            for wk in works:
                wk.wait()
        self._optimizer_step(self.lr if lr is None else lr)
        return self.losses
