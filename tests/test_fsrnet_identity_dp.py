"""Host-side scaling of the identity term on CPU: a world-size-2 gloo run of FSRNetTrainer(identity_net=...) with the
native identity chunk replaced by a deterministic stand-in.  Summed chunk gradients, SUM-reduced across ranks, must
weight every sample's identity term by the global-batch mean, as the single-process step on the concatenated batch does."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.test_dp_gloo import _data, _free_port

W_ID = 0.5


def _make_trainer(world):
    from crfr_b200.model.FSRnet import OverallNetwork, weights_init
    from crfr_b200.model.model_irse import IR_50
    from crfr_b200.trainer import FSRNetTrainer

    class FakeIdTrainer(FSRNetTrainer):
        """Stand-in for crfr_fsrnet_id_train_step: the identity term is a chunk MEAN of per-sample values v_i = mean(hr_i)
        run with id_scale, so grad_k += w_id * id_scale * (k+1) * mean_chunk(v_i); the FSRNet terms as in test_dp_gloo."""

        def _native_chunk(self, *args):
            raise AssertionError("the identity trainer must call _native_id_chunk")

        def _native_id_chunk(self, x, hr, heatmap, labels, outs, loss_div, id_scale, events):
            s = float(x.double().mean(dim=(1, 2, 3)).mean())
            v = float(hr.double().mean(dim=(1, 2, 3)).mean())
            for k, g in enumerate(self.grad_views):
                g.add_(s * (k + 1) / loss_div + self.w_id * id_scale * v * (k + 1))
            self.losses.copy_(torch.tensor([s / loss_div + id_scale * self.w_id * v, 1.0, 2.0, 3.0, 4.0, self.w_id * v]))

        def _optimizer_step(self, lr):
            pass

    torch.manual_seed(1234)
    net = OverallNetwork()
    net.apply(weights_init)
    teacher = IR_50([112, 112]).eval()
    return FakeIdTrainer(net, lr=1e-3, chunk=3, world_size=world, identity_net=teacher, w_id=W_ID)


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        tr = _make_trainer(world)
        x, hr, hm, lbl = _data(8 * world)
        sl = slice(rank * 8, rank * 8 + 8)
        losses = tr.step(x[sl], hr[sl], hm[sl], lbl[sl])
        ret[rank] = (tr.flat_g.clone(), losses.clone())
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_dp2_identity_term_weighs_every_sample_by_the_global_mean():
    world = 2
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    tr = _make_trainer(1)
    x, hr, hm, lbl = _data(8 * world)
    losses = tr.step(x, hr, hm, lbl)
    assert losses.shape == (6,)
    # the identity part of the gradient of parameter k: w_id * (k+1) * (1/G) sum_i v_i over the global batch
    G = x.shape[0]
    v = hr.double().mean(dim=(1, 2, 3))
    s = x.double().mean(dim=(1, 2, 3))
    views = tr.grad_views
    for k in (0, 1, len(views) - 1):
        expect = (k + 1) * (float(s.sum()) / (2.0 * G * G) + W_ID * float(v.sum()) / G)
        assert torch.allclose(views[k].double(), torch.full_like(views[k].double(), expect), rtol=1e-5, atol=1e-9), k
    for r in range(world):
        g, l = ret[r]
        assert torch.allclose(g, tr.flat_g, rtol=1e-5, atol=1e-9)
        # the rank-local parts: the identity entry is the rank's batch mean of w_id * v_i
        assert abs(float(l[5]) - W_ID * float(v[r * 8:r * 8 + 8].mean())) < 1e-6
    # the per-rank totals add up to the global-batch loss, identity term included
    assert abs(sum(float(ret[r][1][0]) for r in range(world)) - float(losses[0])) < 1e-6 * abs(float(losses[0])) + 1e-9
    assert abs(float(losses[5]) - W_ID * float(v.mean())) < 1e-6
