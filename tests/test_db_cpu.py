"""CPU: the DB detector's oracle port (float64) and the refapi SegDetector / L1BalanceCELoss framework path reproduce what the
unmodified reference computes (tests/golden/db_ref.npz, recorded by oracle/make_golden_db.py), and the surfaces carry the
reference's state-dict keys and shapes, including those of the model experiments/seg_detector/seg_detector_db.yaml builds."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import db_port
from oracle.make_golden_db import HEAD_ARGS, LOSS_CASES, head_features
from tests.weights import fill_state_dict

GOLD = os.path.join(os.path.dirname(__file__), "golden", "db_ref.npz")
MAPS = ("binary", "thresh", "thresh_binary")


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLD))


def _case(gold, i):
    p = "loss%d.in." % i
    pred = {k: torch.from_numpy(gold[p + k]).requires_grad_(True) for k in MAPS}
    batch = {k: torch.from_numpy(gold[p + k]) for k in ("gt", "mask", "thresh_map", "thresh_mask")}
    return pred, batch


def _check_loss(gold, i, fn, rtol):
    pred, batch = _case(gold, i)
    loss, metrics = fn(pred, batch)
    grads = torch.autograd.grad(loss, [pred[k] for k in MAPS])
    np.testing.assert_allclose(loss.detach().numpy(), gold["loss%d.loss" % i], rtol=rtol)
    assert sorted(metrics) == ["bce_loss", "l1_loss", "thresh_loss"]
    for k, v in metrics.items():
        np.testing.assert_allclose(v.detach().numpy(), gold["loss%d.metrics.%s" % (i, k)], rtol=rtol)
    for k, g in zip(MAPS, grads):
        r = gold["loss%d.grad.%s" % (i, k)]
        np.testing.assert_allclose(g.numpy(), r, rtol=rtol, atol=rtol * float(np.abs(r).max()))


@pytest.mark.parametrize("i", range(len(LOSS_CASES)))
def test_port_equals_reference_loss_and_gradients(gold, i):
    assert int(gold["loss%d.in.binary" % i].shape[0]) == LOSS_CASES[i][1]
    _check_loss(gold, i, db_port.l1_balance_ce_loss, 1e-12)


@pytest.mark.parametrize("i", range(len(LOSS_CASES)))
def test_port_tie_split_has_the_same_value(gold, i):
    pred, batch = _case(gold, i)
    a, _ = db_port.l1_balance_ce_loss(pred, batch)
    b, _ = db_port.l1_balance_ce_loss(pred, batch, tie_split=True)
    np.testing.assert_allclose(float(a.detach()), float(b.detach()), rtol=1e-14)


def test_port_batches_are_the_recorded_inputs(gold):
    for i, (seed, N, H, W) in enumerate(LOSS_CASES):
        pred, batch = db_port.db_batch(seed, N, H, W, torch.float64)
        for k, v in list(pred.items()) + list(batch.items()):
            np.testing.assert_array_equal(v.numpy(), gold["loss%d.in.%s" % (i, k)])


@pytest.mark.parametrize("i", range(len(LOSS_CASES)))
def test_refapi_loss_on_cpu_equals_reference(gold, i):
    import megreader_b200.refapi.decoders as md
    crit = md.SegDetectorLossBuilder("L1BalanceCELoss").build()
    _check_loss(gold, i, crit, 1e-12)


def test_refapi_head_on_cpu_equals_reference(gold):
    import megreader_b200.refapi.decoders as md
    threads = torch.get_num_threads()
    torch.set_num_threads(1)                              # the summation order of the recording
    try:
        head = fill_state_dict(md.SegDetector(**HEAD_ARGS), "db.")
        feats = head_features()
        with torch.no_grad():
            for mode in ("train", "eval"):
                res = head.train(mode == "train")(feats)
                assert list(res) == list(MAPS)
                for k, v in res.items():
                    np.testing.assert_allclose(v.numpy(), gold["head.%s.%s" % (mode, k)], rtol=1e-5, atol=1e-6)
    finally:
        torch.set_num_threads(threads)


def test_refapi_maps_equal_port():
    import megreader_b200.refapi.decoders as md
    head = md.SegDetector(**HEAD_ARGS)
    torch.manual_seed(0)
    x, y = torch.randn(2, 1, 8, 8), torch.randn(2, 1, 8, 8)
    b, t, tb = db_port.maps(x, y, 50)
    assert torch.equal(head.step_function(b, t), tb)


def test_state_dicts_equal_reference(gold):
    import megreader_b200
    megreader_b200.install_reference_api()                # the deformable trunk imports assets.ops.dcn
    import backbones as mb
    import decoders as md
    keys = json.loads(str(gold["keys_json"]))
    head = md.SegDetector(**HEAD_ARGS)
    assert [[k, list(v.shape)] for k, v in head.state_dict().items()] == keys["SegDetector"]
    y = keys["yaml"]
    assert y["model"] == "SegDetectorModel" and y["model_args"]["loss_class"] == "L1BalanceCELoss"
    model = torch.nn.Module()
    model.backbone = getattr(mb, y["model_args"]["backbone"])(**y["model_args"]["backbone_args"])
    model.decoder = getattr(md, y["model_args"]["decoder"])(**y["model_args"]["decoder_args"])
    assert {k: list(v.shape) for k, v in model.state_dict().items()} == y["state"]
    assert sum(p.numel() for p in model.parameters()) == y["n_params"]


def test_weights_init_matches_reference_rule():
    import megreader_b200.refapi.decoders as md
    head = md.SegDetector(**HEAD_ARGS)
    for name, m in head.named_modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            assert torch.all(m.weight == 1) and torch.all(m.bias == 1e-4), name
    assert head.k == 50 and head.adaptive and not head.serial


def test_smooth_upsampling_fails_like_the_reference():
    import megreader_b200.refapi.decoders as md
    with pytest.raises(TypeError):
        md.SegDetector(adaptive=True, smooth=True)


def test_builder_builds_l1_balance_ce_loss_only():
    import megreader_b200.refapi.decoders as md
    crit = md.SegDetectorLossBuilder("L1BalanceCELoss", eps=1e-6, l1_scale=10, bce_scale=5).build()
    assert isinstance(crit, md.L1BalanceCELoss) and (crit.l1_scale, crit.bce_scale) == (10, 5)
    with pytest.raises(NotImplementedError, match="DiceLoss"):
        md.SegDetectorLossBuilder("DiceLoss").build()
