"""The bf16 reference of the IR_50 input-gradient tests (``tests/test_ir50_grad_gpu.py``) adds gradient roundings to
``oracle.resnet_oracle.ir50_forward``; its forward must stay that oracle's, whose outputs are pinned by the golden
fixture.  CPU only."""
import torch

from tests.test_ir50_grad_gpu import _ir50_ref, _state


def test_ir50_grad_reference_forward_is_the_oracle():
    from oracle import resnet_oracle as RO
    sd = _state()
    x = RO.synthetic_faces(2, seed=4322)
    with torch.no_grad():
        for name in ("fp32", "bf16"):
            pr = RO.Precision(name)
            emb, feats = _ir50_ref(sd, x, pr)
            ref_emb, ref_feats = RO.ir50_forward(sd, x, pr=pr, want_features=True)
            assert torch.equal(emb, ref_emb), name
            assert len(feats) == 4 and all(torch.equal(a, b) for a, b in zip(feats, ref_feats)), name
