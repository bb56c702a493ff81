"""Host-side checks of the SUPER_RESOLUTION variant's modules (crfr_b200/SUPER_RESOLUTION/model/FSRnet.py) that need no
GPU: the native program runs the reference's default configuration only, and a module built with other constructor
arguments is refused before anything reaches the device, even where its parameter count matches the default one."""
import pytest
import torch


def _cases():
    from crfr_b200.SUPER_RESOLUTION.model import FSRnet as M
    return [(M.Coarse_SR_Network, dict(ngf=32), 3), (M.Fine_SR_Encoder, dict(ngf=32), 3),
            (M.Prior_Estimation_Network, dict(parsing_classes=11, num_landmark=5), 3),
            (M.Fine_SR_Decoder, dict(ngf=64), 64), (M.Coarse_SR_Network, dict(n_blocks=4), 3)]


def test_non_default_modules_are_refused_before_any_launch():
    from crfr_b200.SUPER_RESOLUTION.model import FSRnet as M
    for cls, kwargs, cin in _cases():
        m = cls(**kwargs)
        default = len(cls().state_dict())
        if "n_blocks" not in kwargs:                    # the count alone would not have caught these
            assert len(m.state_dict()) == default, (cls.__name__, kwargs)
        with pytest.raises(NotImplementedError, match="default configuration"):
            m(torch.randn(1, cin, 32, 32))              # a CPU tensor: the refusal comes first, nothing is launched
    M.check_parameter_table(M.Fine_SR_Encoder(), list(M.Fine_SR_Encoder().state_dict().values()))


def test_default_modules_keep_the_cpu_error():
    from crfr_b200.SUPER_RESOLUTION.model.FSRnet import Coarse_SR_Network
    with pytest.raises(RuntimeError, match="CUDA"):
        Coarse_SR_Network()(torch.randn(1, 3, 32, 32))
