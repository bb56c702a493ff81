"""bench.py --dump-outputs at the benchmark's own sizes (batch 128, 128 x 128): file set, dtype, the 64 MB bound and a
sample that is the same from run to run.  The trainer's arenas and output buffers live on the host here; the dump reads
them the same way on the device."""
import os

import numpy as np
import torch

import bench

NAMES = ("losses", "params", "grads", "out_coarse", "out_sr", "out_landmark", "out_parsing")


def _trainer(batch):
    from crfr_b200.model import FSRnet as M
    from crfr_b200.trainer import FSRNetTrainer
    torch.manual_seed(1234)
    net = M.OverallNetwork()
    net.apply(M.weights_init)
    tr = FSRNetTrainer(net, chunk=batch)
    g = torch.Generator().manual_seed(0)
    tr.flat_g.copy_(torch.randn(tr.total, generator=g))
    tr.outs = tuple(torch.randn(t.shape, generator=g) for t in M.alloc_outputs(torch.empty(batch, 3, 128, 128)))
    return tr


def test_dump_outputs_at_bench_size(tmp_path):
    batch = 128
    tr = _trainer(batch)
    losses = torch.tensor([5.0, 1.0, 2.0, 3.0, 4.0])
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), tr, losses, batch)
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in NAMES)
    total = 0
    for n in NAMES:
        a, b = np.load(tmp_path / "a" / (n + ".npy")), np.load(tmp_path / "b" / (n + ".npy"))
        assert a.dtype == np.float32 and np.array_equal(a, b), n
        total += os.path.getsize(tmp_path / "a" / (n + ".npy"))
    assert total <= 64e6, total
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "losses.npy"), losses.numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "params.npy"), tr.flat_p.numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "grads.npy"), tr.flat_g.numpy())
    for n, t in zip(NAMES[3:], tr.outs):
        s = np.load(tmp_path / "a" / (n + ".npy"))
        assert s.shape == (bench.OUTPUT_SAMPLE,) and np.isin(s, t.numpy()).all(), n


def test_dump_outputs_without_whole_batch_outputs(tmp_path):
    """With several chunks per step the trainer keeps only the last chunk's outputs: the dump leaves them out."""
    tr = _trainer(4)
    bench.dump_outputs(str(tmp_path), tr, torch.zeros(5), 8)
    assert sorted(os.listdir(tmp_path)) == ["grads.npy", "losses.npy", "params.npy"]
