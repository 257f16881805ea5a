"""GPU: the DB detector's kernels (csrc/db_head.cu through megreader_b200/db.py and the refapi surfaces) against the float64
oracle port (oracle/db_port.py): loss, metrics and the gradients of all four outputs, edge cases of the balanced selection,
determinism, CUDA-graph replay, the memory bound, and the training step on the engine against the fp32 library path."""
import numpy as np
import pytest
import torch

from oracle import db_port

pytestmark = pytest.mark.gpu

MAPS = ("binary", "thresh", "thresh_binary")
LABELS = ("gt", "mask", "thresh_map", "thresh_mask")
COEF = (1.0, 0.3, -0.7, 0.2)            # upstream gradients of (loss, bce_loss, thresh_loss, l1_loss)


def _kernel(pred, batch, dev):
    from megreader_b200 import db
    leaves = [pred[k].to(dev, torch.float32).contiguous().requires_grad_(True) for k in MAPS]
    lab = [batch[k].to(dev, torch.float32).contiguous() for k in LABELS]
    out = db.l1_balance_ce_loss(*leaves, *lab)
    (out * torch.tensor(COEF, device=dev)).sum().backward()
    return out.detach().cpu().double(), [x.grad.cpu().double() for x in leaves]


def _port(pred, batch, tie_split=True):
    leaves = {k: pred[k].double().cpu().requires_grad_(True) for k in MAPS}
    lab = {k: batch[k].double().cpu() for k in LABELS}
    loss, m = db_port.l1_balance_ce_loss(leaves, lab, tie_split=tie_split)
    out = torch.stack([loss, m["bce_loss"], m["thresh_loss"], m["l1_loss"]])
    grads = torch.autograd.grad((out * torch.tensor(COEF, dtype=torch.float64)).sum(), [leaves[k] for k in MAPS])
    return out.detach(), list(grads)


def _tau(pred, batch):
    """The selection threshold (k-th largest negative BCE entry) and k, from the literal float64 composition."""
    b, g, m = pred["binary"].double(), batch["gt"].double(), batch["mask"].double()
    neg = ((1 - g) * m).byte()
    pos = int((g * m).byte().float().sum())
    k = min(int(neg.float().sum()), int(pos * 3.0))
    loss = torch.nn.functional.binary_cross_entropy(b, g, reduction="none")[:, 0]
    if k == 0:
        return None, 0, loss
    return float(torch.topk((loss * neg.double()).view(-1), k)[0][-1]), k, loss


def _compare(pred, batch, dev, rtol=2e-5, exclude_near_tau=True):
    out_k, g_k = _kernel(pred, batch, dev)
    out_p, g_p = _port(pred, batch)
    np.testing.assert_allclose(out_k.numpy(), out_p.numpy(), rtol=rtol, atol=1e-7, equal_nan=True)
    keep = torch.ones_like(pred["binary"], dtype=torch.bool)
    if exclude_near_tau:
        tau, _, loss = _tau(pred, batch)
        if tau is not None:
            keep = ((loss - tau).abs() > 1e-5 * max(tau, 1e-30)).unsqueeze(1)
    for name, a, r in zip(MAPS, g_k, g_p):
        sel = keep if name == "binary" else torch.ones_like(keep)
        scale = float(r[sel].abs().max()) if bool(torch.isfinite(r[sel]).all()) else 1.0
        np.testing.assert_allclose(a[sel].numpy(), r[sel].numpy(), rtol=rtol, atol=rtol * scale, equal_nan=True, err_msg=name)
    return out_k, g_k


def test_case_a_single_sample(cuda):
    _compare(*db_port.db_batch(11, 1, 64, 80), cuda)


def test_case_b_three_samples_non_square_with_ignore_regions(cuda):
    pred, batch = db_port.db_batch(12, 3, 48, 72)
    assert float(batch["mask"].min()) == 0.0
    _compare(pred, batch, cuda)


def test_case_c_quantised_predictions_ties(cuda):
    pred, batch = db_port.db_batch(13, 3, 40, 56)
    pred["binary"] = (torch.round(pred["binary"] * 256) / 256).clamp(1 / 256, 255 / 256)
    tau, k, loss = _tau(pred, batch)
    negc = int(((1 - batch["gt"].double()) * batch["mask"].double()).byte().float().sum())
    assert tau is not None and 0 < k < negc
    # ties at tau are certain; the selection is the same in fp32 and fp64: no element is excluded
    out_k, g_k = _compare(pred, batch, cuda, exclude_near_tau=False)
    tied = (loss == tau).unsqueeze(1)
    assert int(tied.sum()) > 1
    # literal topk puts the tied remainder r on some of the tied copies, the kernels spread it evenly: same loss, and the
    # summed gradient over the tied set is the same (every tied copy has the same b and g = 0)
    out_lit, g_lit = _port(pred, batch, tie_split=False)
    np.testing.assert_allclose(out_k.numpy(), out_lit.numpy(), rtol=2e-5)
    np.testing.assert_allclose(float(g_k[0][tied].sum()), float(g_lit[0][tied].sum()), rtol=2e-5)


def test_case_d_no_positives(cuda):
    pred, batch = db_port.db_batch(14, 2, 32, 40)
    batch["gt"].zero_()
    assert _tau(pred, batch)[1] == 0
    out_k, g_k = _compare(pred, batch, cuda)
    assert float(out_k[1]) == 0.0 and float(g_k[0].abs().max()) == 0.0


def test_case_e_k_capped_by_negatives(cuda):
    pred, batch = db_port.db_batch(15, 2, 32, 40)
    batch["gt"].fill_(1.0)
    batch["gt"][:, :, :3, :5] = 0.0
    _, k, _ = _tau(pred, batch)
    negc = int(((1 - batch["gt"]) * batch["mask"]).byte().float().sum())
    assert k == negc > 0
    _compare(pred, batch, cuda)


def test_case_f_binary_exactly_zero_and_one(cuda):
    pred, batch = db_port.db_batch(16, 2, 32, 40)
    b = pred["binary"]
    b[:, :, :4, :] = 0.0
    b[:, :, 4:8, :] = 1.0
    batch["gt"][:, :, :2, :] = 1.0          # b = 0, g = 1: log clamped at -100
    batch["gt"][:, :, 4:6, :] = 0.0         # b = 1, g = 0: log1p clamped at -100, (1 - b) b under 1e-12
    _compare(pred, batch, cuda)


def test_case_g_half_values_truncate(cuda):
    pred, batch = db_port.db_batch(17, 3, 32, 40)
    batch["gt"][0, 0, :8, :] = 0.5
    batch["mask"][1, 8:16, :] = 0.5
    _compare(pred, batch, cuda)


def test_case_h_empty_thresh_mask_is_nan(cuda):
    pred, batch = db_port.db_batch(18, 2, 24, 32)
    batch["thresh_mask"].zero_()
    out_k, _ = _compare(pred, batch, cuda)
    assert np.isnan(float(out_k[0])) and np.isnan(float(out_k[3]))


def test_maps_match_framework_autograd(cuda):
    from megreader_b200 import db
    torch.manual_seed(0)
    xb, xt = torch.randn(3, 1, 40, 56, device=cuda) * 3, torch.randn(3, 1, 40, 56, device=cuda)
    gs = [torch.randn(3, 1, 40, 56, device=cuda) for _ in range(3)]
    got, ref = [], []
    for fn, out in ((db.maps, got), (db_port.maps, ref)):
        a, c = xb.clone().requires_grad_(True), xt.clone().requires_grad_(True)
        maps = fn(a, c, 50)
        sum((m * g).sum() for m, g in zip(maps, gs)).backward()
        out += [m.detach() for m in maps] + [a.grad, c.grad]
    for a, r in zip(got, ref):
        torch.testing.assert_close(a, r, rtol=1e-5, atol=1e-6)


def test_loss_is_deterministic(cuda):
    pred, batch = db_port.db_batch(19, 4, 96, 128)
    o1, g1 = _kernel(pred, batch, cuda)
    o2, g2 = _kernel(pred, batch, cuda)
    assert torch.equal(o1, o2) and all(torch.equal(a, b) for a, b in zip(g1, g2))


def test_cuda_graph_replay_equals_eager(cuda):
    from megreader_b200 import db
    batches = [db_port.db_batch(s, 3, 64, 64) for s in (20, 21)]
    static = {k: v.to(cuda, torch.float32).contiguous() for k, v in list(batches[0][0].items()) + list(batches[0][1].items())}
    leaves = [static[k].requires_grad_(True) for k in MAPS]
    coef = torch.tensor(COEF, device=cuda)

    def run():
        for x in leaves:
            x.grad = None
        out = db.l1_balance_ce_loss(*leaves, *[static[k] for k in LABELS])
        (out * coef).sum().backward()
        return out
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            run()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = run()
    pred, batch = batches[1]
    with torch.no_grad():
        for k, v in list(pred.items()) + list(batch.items()):
            static[k].copy_(v.to(cuda, torch.float32))
    graph.replay()
    torch.cuda.synchronize()
    o_e, g_e = _kernel(pred, batch, cuda)
    assert torch.equal(static_out.detach().cpu().double(), o_e)
    for x, r in zip(leaves, g_e):
        assert torch.equal(x.grad.cpu().double(), r)


def test_peak_memory_at_yaml_batch(cuda):
    import bench_db
    from megreader_b200 import db
    N, H, W = 16, 640, 640
    pred, batch = bench_db.loss_inputs(3, N, H, W, cuda)
    leaves = [pred[k].detach().requires_grad_(True) for k in MAPS]
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = db.l1_balance_ce_loss(*leaves, *[batch[k] for k in LABELS])
    out[0].backward()
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    # workspace (<= 16 B per sample-pixel + O(grid)) and the three gradients (12 B per sample-pixel)
    assert extra <= (16 + 12) * N * H * W + (4 << 20), extra
    assert extra < 0.5 * 4 * N * N * H * W                # one fp32 (N,N,H,W) temporary of the reference: 420 MB
    assert bool(torch.isfinite(out).all())


def test_refapi_surfaces_run_the_kernels(cuda):
    import megreader_b200.refapi.decoders as md
    from megreader_b200 import _lib
    from oracle.make_golden_db import HEAD_ARGS, head_features
    from tests.weights import fill_state_dict
    head = fill_state_dict(md.SegDetector(**HEAD_ARGS), "db.").to(cuda).train()
    feats = [f.to(cuda) for f in head_features()]
    _lib.reset_launch_count()
    pred = head(feats)
    ref = head._forward_framework(head._fuse(feats))
    for k in MAPS:
        torch.testing.assert_close(pred[k], ref[k], rtol=1e-5, atol=1e-5)
    n, _, h, w = pred["binary"].shape
    _, batch = db_port.db_batch(3, n, h, w)
    batch = {k: v.to(cuda) for k, v in batch.items()}
    loss, metrics = md.L1BalanceCELoss()(pred, batch)
    loss.backward()
    assert _lib.launch_count() >= 1 + 9 + 1 + 1
    ref_loss, ref_m = db_port.l1_balance_ce_loss({k: v.detach().double().cpu() for k, v in pred.items()},
                                                 {k: v.double().cpu() for k, v in batch.items()})
    np.testing.assert_allclose(float(loss), float(ref_loss), rtol=2e-5)
    for k, v in metrics.items():
        np.testing.assert_allclose(float(v), float(ref_m[k]), rtol=2e-5)
    assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in head.parameters())


def test_db_step_engine_vs_library(cuda):
    """deformable_resnet50 + SegDetector + L1BalanceCELoss: the engine (bf16 tcgen05 convolutions + the DB kernels) against the fp32
    modules with the literal loss; same loss and gradient-direction thresholds as tests/test_trunks_engine_gpu.py."""
    import bench_db
    from oracle import db_port as port
    torch.manual_seed(0)
    net = bench_db.build_model(cuda, engine=False)
    for m in net.modules():                      # running statistics, as in tests/test_trunks_engine_gpu.py
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eval()
    batch = bench_db.synth_batch(5, 2, 256, 256, cuda)
    import decoders
    crit = decoders.L1BalanceCELoss()

    def run(engine):
        for p in net.parameters():
            p.grad = None
        if engine:
            loss, _ = crit(net(batch["image"]), batch)
        else:
            loss, _ = port.l1_balance_ce_loss(net.forward_library(batch["image"]), batch)
        loss.backward()
        return float(loss), {n: p.grad.detach().float().clone() for n, p in net.named_parameters() if p.grad is not None}
    loss_ref, g_ref = run(False)
    from megreader_b200 import conv_engine
    assert conv_engine.use_engine_convs(net) > 40
    try:
        loss_eng, g_eng = run(True)
    finally:
        conv_engine.restore_library_convs(net)
    assert abs(loss_eng - loss_ref) / abs(loss_ref) < 5e-2, (loss_eng, loss_ref)
    assert all(torch.isfinite(v).all() for v in g_eng.values())
    assert set(g_eng) == set(g_ref)
    checked = 0
    for n, r in g_ref.items():
        if r.numel() >= 64 * 64 and float(r.norm()) > 1e-6:
            cos = float((r * g_eng[n]).sum() / (r.norm() * g_eng[n].norm() + 1e-20))
            assert cos > 0.9, (n, cos)
            checked += 1
    assert checked > 20
