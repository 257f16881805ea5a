"""CPU: the ATen-composed surfaces of megreader_b200.refapi (SURVEY.md §8 A9/A10) reproduce the reference goldens and carry
the reference's exact state-dict keys/shapes, deformable trunk included."""
import gzip
import json
import os

import numpy as np
import pytest
import torch

from tests import surfaces_common as sc
from tests.weights import east_inputs, fill_state_dict

STATE_GOLD = os.path.join(os.path.dirname(__file__), "golden", "state_dicts_ref.json.gz")
EAST_GOLD = os.path.join(os.path.dirname(__file__), "golden", "east_ref.npz")


def test_backbones_reproduce_reference_golden():
    torch.set_num_threads(4)
    sc.check_backbones("cpu", 1e-5)


def test_attention_head_reproduces_reference_golden():
    sc.check_attention("cpu", 2e-5)


def test_ctc_conv_head_eval_reproduces_reference_golden():
    sc.check_ctc_head("cpu", 1e-5, train=False)


def test_ctc_conv_head_train_refuses_cpu():
    with pytest.raises(NotImplementedError):
        sc.check_ctc_head("cpu", 1e-5, train=True)


def _keys(m):
    return [[k, list(v.shape)] for k, v in m.state_dict().items()]


def test_state_dict_keys_equal_reference():
    """Keys and shapes equal those of the reference's modules, recorded by `python -m oracle.make_golden state_dicts`."""
    import sys
    import types
    import megreader_b200.refapi.backbones as mb
    import megreader_b200.refapi.decoders as md
    import megreader_b200.refapi.backbones.resnet as mres
    from megreader_b200 import dcn as mdcn
    with gzip.open(STATE_GOLD, "rt") as f:
        ref = json.load(f)["modules"]
    mine = {"resnet34": mb.resnet34(pretrained=False), "resnet101": mb.resnet101(pretrained=False),
            "Resnet34FPN": mb.Resnet34FPN(resnet_pretrained=False),
            "resnet50dilated_ppm": mb.resnet50dilated_ppm(inner_channels=128),
            "AttentionDecoder": md.AttentionDecoder(64, inner_channels=128, max_size=16, height=2),
            "CTCDecoder": md.CTCDecoder(64, inner_channels=96), "EASTDecoder": md.EASTDecoder(channels=64)}
    # deformable trunk: our modules resolve `assets.ops.dcn` lazily; bind it to megreader_b200.dcn for this process
    shim = types.ModuleType("assets.ops.dcn")
    shim.ModulatedDeformConv, shim.DeformConv = mdcn.ModulatedDeformConv, mdcn.DeformConv
    saved = sys.modules.get("assets.ops.dcn")
    sys.modules["assets.ops.dcn"] = shim
    try:
        mine["deformable_resnet50"] = mres.deformable_resnet50(pretrained=False)
        mine["ResNet_v1_dcn"] = mres.ResNet(mres.BasicBlock, [1, 1, 1, 1], dcn=dict(modulated=False, deformable_groups=2))
    finally:
        if saved is not None:
            sys.modules["assets.ops.dcn"] = saved
        else:
            del sys.modules["assets.ops.dcn"]
    # deformable RoI pooling packs: same fully-connected stacks
    from megreader_b200 import deform_pool as mpool
    for cls in ("DeformRoIPoolingPack", "ModulatedDeformRoIPoolingPack"):
        mine[cls] = getattr(mpool, cls)(0.5, 3, 8, False, trans_std=0.1, deform_fc_channels=32)
    assert sorted(mine) == sorted(ref)
    for name, m in mine.items():
        assert _keys(m) == ref[name], name
    # zero-initialised offset branch (resnet.py:222-226)
    for mod in mine["deformable_resnet50"].modules():
        if hasattr(mod, "conv2_offset"):
            assert float(mod.conv2_offset.weight.abs().max()) == 0.0 and float(mod.conv2_offset.bias.abs().max()) == 0.0
    # dilation surgery moved the same convs (resnet_dilated.py:37-49)
    geo = [[n, list(c.stride), list(c.dilation), list(c.padding)] for n, c in mb.resnet50dilated_ppm().named_modules()
           if isinstance(c, torch.nn.Conv2d)]
    with gzip.open(STATE_GOLD, "rt") as f:
        assert geo == json.load(f)["resnet50dilated_ppm_conv_geometry"]


def test_east_decoder_equals_reference_module():
    """decoders/east.py:7-60 on CPU: same parameters -> the reference module's loss, metrics and predictions (train and eval
    branches), recorded by `python -m oracle.make_golden east` with one host thread."""
    import megreader_b200.refapi.decoders as md
    g = np.load(EAST_GOLD)
    m = fill_state_dict(md.EASTDecoder(channels=32), "east.").train()
    torch.set_num_threads(1)
    x, label = east_inputs()
    lm, pm, mm = m(x, label, None, True)
    torch.testing.assert_close(lm, torch.from_numpy(g["loss"]))
    for prefix, got in (("pred.", pm), ("metrics.", mm)):
        assert sorted(prefix + k for k in got) == sorted(k for k in g.files if k.startswith(prefix))
        for k in got:
            torch.testing.assert_close(got[k], torch.from_numpy(g[prefix + k]))
    m.eval()
    pe_m = m(x, label, None, False)
    assert sorted("eval." + k for k in pe_m) == sorted(k for k in g.files if k.startswith("eval."))
    for k in pe_m:
        torch.testing.assert_close(pe_m[k], torch.from_numpy(g["eval." + k]))
