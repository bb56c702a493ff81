"""Host-side checks that need no GPU: the C-ABI library builds/loads, exports every symbol include/crfr.h declares,
the host-only entry points work, and the Python mirror keeps the reference's interface."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import crfr_b200
    crfr_b200.build()
    from crfr_b200 import _lib
    return _lib.lib()


def test_library_exports_every_declared_symbol(lib):
    from crfr_b200 import _lib
    header = open(os.path.join(ROOT, "include", "crfr.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(crfr_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 38
    for name in sorted(declared):
        assert hasattr(lib, name), "libcrfr.so does not export %s" % name
        assert name in _lib.SIGNATURES, "no ctypes signature for %s" % name
    assert set(_lib.SIGNATURES) == declared
    assert lib.crfr_version() >= 100


def test_integration_doc_lists_every_entry_point():
    """INTEGRATION.md's appendix (tools/abi_table.py) names every declared entry point next to the reference interface it
    stands in for."""
    header = open(os.path.join(ROOT, "include", "crfr.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(crfr_[a-z0-9_]+)\s*\(", header))
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    listed = set(re.findall(r"^\| `(crfr_[a-z0-9_]+)` \|", doc, flags=re.M))
    assert listed == declared, (sorted(declared - listed), sorted(listed - declared))


def test_struct_layouts_match_header():
    from crfr_b200 import _lib
    assert C.sizeof(_lib.ConvDesc) == 13 * 4
    assert C.sizeof(_lib.FsrnetIO) == 8 + 8 * 8 + 8 + 3 * 8      # 2 ints, 8 pointers, 2 floats, 3 event handles
    assert _lib.FSRNET_NPARAMS == 202


def test_error_convention(lib):
    from crfr_b200 import _lib
    rc = lib.crfr_bicubic_tables(0, 8, None)
    assert rc != 0 and b"bicubic_tables" in lib.crfr_last_error()
    with pytest.raises(RuntimeError, match="bicubic_tables"):
        _lib.call("crfr_bicubic_tables", 16, 128, None)
    assert lib.crfr_fsrnet_workspace_bytes(4, 100, 1) == 0          # size must be a multiple of 16


def test_set_option_names(lib):
    """crfr_set_option takes the five implementation switches at their defaults and rejects the retired ones by name."""
    for name in ("rowconv_pair", "wgrad_stream", "norm_bwd_impl", "norm_fwd_stream", "fuse_norm_bwd"):
        assert lib.crfr_set_option(name.encode(), 1) == 0, lib.crfr_last_error()
    for name in ("rowconv", "pair_swap", "rowwgrad_pair", "fuse_norm_fwd", "pdl", "tc_t2", "bn_fused_stats",
                 "matcher_cluster", "pair_debug", "ir50_stem_tc"):
        assert lib.crfr_set_option(name.encode(), 0) == 1                # CRFR_EINVAL
        assert ("'%s'" % name).encode() in lib.crfr_last_error()


def test_bicubic_tables_match_oracle(lib):
    from crfr_b200 import ops
    from oracle import bicubic_oracle as BO
    for s, o in ((16, 128), (28, 224), (20, 50), (7, 7), (64, 16)):
        tab = ops.bicubic_table_host(s, o)
        xmin, cnt, kk = BO.coeff_table(s, o)
        assert np.array_equal(tab[:, 0], xmin) and np.array_equal(tab[:, 1], cnt)
        assert np.array_equal(tab[:, 2:2 + kk.shape[1]], kk)


def test_rotate_coeffs_match_oracle(lib):
    """crfr_rotate_coeffs (C: cos / sin rounded to 15 decimals through the decimal string, 16.16 FIX) against the Python
    restatement of Pillow's Image.rotate matrix - the host part of the augmentation, no GPU needed."""
    import ctypes as C
    import random
    from oracle import augment_oracle as AO
    rng = random.Random(3)
    buf = (C.c_int32 * 6)()
    cases = [(28, 28, 0.0), (28, 28, 360.0), (112, 112, -10.0), (224, 224, 10.0), (33, 40, 180.0), (17, 5, -725.5)]
    cases += [(rng.choice([28, 112, 128, 224, 31]), rng.choice([28, 112, 128, 224, 57]), rng.uniform(-400, 400))
              for _ in range(500)]
    for h, w, ang in cases:
        assert lib.crfr_rotate_coeffs(h, w, ang, C.cast(buf, C.c_void_p)) == 0
        assert list(buf) == AO.rotate_coeffs(h, w, ang).tolist(), (h, w, ang)


def test_workspace_sizing_is_monotonic(lib):
    a = lib.crfr_fsrnet_workspace_bytes(2, 64, 1)
    b = lib.crfr_fsrnet_workspace_bytes(4, 64, 1)
    c = lib.crfr_fsrnet_workspace_bytes(4, 64, 0)
    assert 0 < c < b and a < b < 2.2 * a


def test_tcgen05_shape_support_table(lib):
    from crfr_b200 import _lib
    sup = lambda op, h, cin, cout, k=3, s=1, p=1: bool(lib.crfr_conv_engine_supported(_lib.ENGINE_TCGEN05, op, h, h, cin, cout, k, s, p))
    for op in (0, 1, 2):
        assert sup(op, 128, 64, 64) and sup(op, 32, 128, 128) and sup(op, 8, 128, 128) and sup(op, 32, 192, 64)
    # edge layers ride the tensor cores through the lowered (im2col + GEMM) recipes
    assert sup(0, 128, 3, 64) and sup(2, 128, 3, 64) and not sup(1, 128, 3, 64)
    assert sup(0, 128, 64, 3) and sup(1, 128, 64, 3) and sup(0, 128, 3, 64, 7, 4, 3) and sup(1, 128, 3, 128, 7, 4, 3)
    assert not sup(0, 32, 128, 11, 1, 1, 0) and sup(0, 100, 64, 64) and sup(2, 100, 64, 64)
    # ResNet_34 trunk (model/resnet.py): wide layers use several column tiles, partial pixel tiles are zero filled,
    # the stage transitions (3x3 s2, 1x1 s2) and the 7x7 s2 stem go through the lowered recipes
    for op in (0, 1, 2):
        assert sup(op, 56, 64, 64) and sup(op, 28, 128, 128) and sup(op, 14, 256, 256) and sup(op, 7, 512, 512)
        assert sup(op, 56, 64, 128, 3, 2, 1) and sup(op, 28, 128, 256, 1, 2, 0) and sup(op, 14, 256, 512, 3, 2, 1)
    assert sup(0, 112, 3, 64, 7, 2, 3) and sup(2, 112, 3, 64, 7, 2, 3)


def test_module_mirror_keeps_reference_interface():
    from crfr_b200.model.FSRnet import OverallNetwork, weights_init
    from oracle import fsrnet_oracle as FO
    torch.manual_seed(1234)
    net = OverallNetwork()
    net.apply(weights_init)
    sd = net.state_dict()
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == [(k, tuple(s)) for k, s in FO.fsrnet_param_shapes()]
    ref = FO.build_fsrnet_state_dict(1234)
    assert all(torch.equal(sd[k], ref[k]) for k in ref)               # identical seeded init, draw for draw
    for name in ("_coarse_sr_network", "_prior_estimation_network", "_fine_sr_encoder", "_fine_sr_decoder"):
        assert hasattr(net, name)                                     # used by name at FSR_main.py:146,158-159
    assert [k for k, _ in net.named_parameters()] == list(sd.keys())


def test_resnet_mirror_keeps_reference_interface():
    from crfr_b200.model.resnet import ResNet_34, ResNet, BasicBlock
    from oracle import resnet_oracle as RO
    torch.manual_seed(77)
    net = ResNet_34()
    sd = net.state_dict()
    ref = RO.build_resnet34_state_dict(77)
    assert list(sd.keys()) == list(ref.keys())
    assert all(torch.equal(sd[k], ref[k]) for k in ref)               # identical seeded init, draw for draw
    assert len(list(net.named_parameters())) == 114 and len(list(net.named_buffers())) == 3 * 38
    with pytest.raises(AssertionError):
        ResNet([96, 96], BasicBlock, [3, 4, 6, 3])                     # model/resnet.py:156
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(1, 3, 112, 112))


def test_ir50_mirror_keeps_reference_interface():
    from crfr_b200.model.model_irse import IR_50, Backbone
    from oracle import resnet_oracle as RO
    torch.manual_seed(91)
    net = IR_50([112, 112])
    sd, ref = net.state_dict(), RO.build_ir50_state_dict(91)
    assert list(sd.keys()) == list(ref.keys()) and all(torch.equal(sd[k], ref[k]) for k in ref)
    assert len(list(net.named_parameters())) == 187 and len(list(net.named_buffers())) == 3 * 54
    with pytest.raises(AssertionError):
        Backbone([96, 96], 50, "ir")                                   # model_irse.py:132
    net.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(1, 3, 112, 112))


def test_product_fails_loudly_without_gpu():
    from crfr_b200.model.FSRnet import OverallNetwork
    from crfr_b200 import ops
    net = OverallNetwork()
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(1, 3, 64, 64))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.nchw_to_nhwc(torch.zeros(1, 3, 8, 8))


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "cross-resolution-face-recognition_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, os.path.join(dp, f)
