"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

Run:  python -m oracle.make_golden            (from the repo root; needs /root/reference)

2D-CTC: the reference's CUDA op cannot run here (no GPU, does not build on torch 2.11), so the
golden vectors come from the reference's own pure-Python CTCLoss2D (decoders/ctc_loss2d.py:86-154)
with (mask + classify) == log_probs, on cases where it does not numerically saturate
(SURVEY.md §8c: valid while every per-state height-sum stays above fp32 tiny, i.e. loss <~ 60).

Targets: ctc2d (default), crnn, surfaces, head, input, crnn_port, state_dicts, east run the reference on the CPU;
ref_kernels runs its compiled CUDA ops (`python -m oracle.build_ref` first) on a GPU.
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def ctc2d_case(seed, T, H, N, C, S, Lmax, peak):
    g = torch.Generator().manual_seed(seed)
    tl = torch.randint(1, Lmax + 1, (N,), generator=g)
    targets = torch.zeros(N, S, dtype=torch.long)
    for b in range(N):
        targets[b, :tl[b]] = torch.randint(1, C, (int(tl[b]),), generator=g)
    il = torch.full((N,), T, dtype=torch.long)
    mask_logit = torch.randn(T, H, N, generator=g)
    cls_logit = torch.randn(T, H, N, C, generator=g)
    if peak > 0:
        # push the classifier toward a monotone alignment of the target so the loss stays small
        for b in range(N):
            L = int(tl[b])
            for t in range(T):
                k = min(L - 1, t * L // T)
                cls_logit[t, :, b, targets[b, k]] += peak
    mask = mask_logit.log_softmax(1)
    classify = cls_logit.log_softmax(3)
    return mask, classify, targets, il, tl


def make_ctc2d():
    m = ref_loader.load("decoders.ctc_loss2d")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = m.CTCLoss2D(blank=0, reduction="none")
    cases = [  # name, seed, T, H, N, C, S, Lmax, peak
        ("doc", 1, 32, 8, 16, 20, 20, 6, 4.0),      # docstring shape decoders/ctc_loss2d.py:37-45 (short targets)
        ("small", 2, 8, 4, 4, 6, 5, 3, 0.0),
        ("cfg3", 3, 32, 8, 8, 38, 32, 5, 5.0),      # res50-ppm-2d-ctc.yaml shape, peaked
        ("h1", 4, 12, 1, 3, 7, 6, 4, 2.0),          # H=1 degenerates to 1D CTC
        ("rep", 5, 16, 3, 4, 5, 8, 6, 3.0),         # tiny alphabet -> repeated labels (have_three false)
    ]
    for name, seed, T, H, N, C, S, Lmax, peak in cases:
        mask, classify, targets, il, tl = ctc2d_case(seed, T, H, N, C, S, Lmax, peak)
        classify.requires_grad_(True)
        loss = ref(mask, classify, targets, il, tl)
        # autograd of the reference python loss = TRUE derivative -exp(G + nll - lp); the CUDA op's K3
        # returns exp(lp) + that on in-target classes (SURVEY.md App. B1.1), which tests check.
        (ref_grad,) = torch.autograd.grad(loss.sum(), classify)
        classify = classify.detach()
        lp = (mask.unsqueeze(-1) + classify).contiguous()
        np.savez_compressed(
            os.path.join(GOLD, "ctc2d_pyref_%s.npz" % name),
            log_probs=lp.numpy(), targets=targets.numpy(), input_lengths=il.numpy(),
            target_lengths=tl.numpy(), ref_nll=loss.detach().numpy(),
            ref_autograd=ref_grad.numpy())
        print("ctc2d", name, "ref nll", loss.detach().numpy()[:4])


def make_crnn():
    """cfg 1 exactly (crnn.yaml): reference crnn_backbone + CRNNDecoder(nn.CTCLoss), N=4, 3x32x100, fp32, CPU."""
    from tests.weights import crnn_batch, fill_state_dict
    ref_loader.install()
    import backbones as rb
    import decoders as rd
    torch.manual_seed(0)
    bb = fill_state_dict(rb.crnn_backbone(), "bb.")
    dec = fill_state_dict(rd.CRNNDecoder(in_channels=512, inner_channels=256), "dec.")
    for name, (N, W) in {"cfg1": (4, 100), "w128": (3, 128)}.items():
        T = W // 4 + 1
        x, labels, lengths = crnn_batch(0, N, W, 8, T)
        bb.train(); dec.train()
        bb.zero_grad(); dec.zero_grad()
        tx = torch.from_numpy(x)
        feat = bb(tx)
        loss, pred = dec(feat, targets=torch.from_numpy(labels), lengths=torch.from_numpy(lengths), train=True)
        loss.mean().backward()
        grads = {"grad." + k: v.grad.numpy().copy() for k, v in list(bb.named_parameters()) + list(dec.named_parameters())
                 if k in ("cnn.0.0.0.weight", "cnn.2.1.weight", "cnn.6.1.bias", "cnn.6.0.bias",
                          "rnn.1.embedding.weight", "rnn.1.embedding.bias", "rnn.0.rnn.bias_hh_l0_reverse")}
        gnorm = {"gnorm." + k: np.float64(v.grad.double().norm().item())
                 for k, v in list(bb.named_parameters()) + list(dec.named_parameters())}
        bn_after = {"bn." + k: v.numpy().copy() for k, v in bb.state_dict().items() if "running" in k and k.startswith("cnn.2")}
        # eval-mode forward AFTER the training forward (running stats updated once), like eval.py would see
        bb.eval(); dec.eval()
        with torch.no_grad():
            prob = dec(bb(tx), train=False)                       # (N, C, 1, T) softmax
        # re-load pristine weights for the next case (BN running stats were updated)
        np.savez_compressed(os.path.join(GOLD, "crnn_ref_%s.npz" % name), x=x[:, :1], labels=labels, lengths=lengths,
                            feature=feat.detach().numpy(), loss=np.float64(loss.item()), log_probs=pred.detach().numpy(),
                            eval_prob=prob.numpy(), **grads, **gnorm, **bn_after)
        print("crnn", name, "loss", loss.item(), "feat", tuple(feat.shape), "pred", tuple(pred.shape))
        fill_state_dict(bb, "bb."); fill_state_dict(dec, "dec.")


def make_surfaces():
    """Recognition-side surfaces around the hot path (SURVEY.md §8 A9/A10 + the 1-D CTC conv head): outputs of the
    UNMODIFIED reference modules on CPU, fp32, weights from tests.weights.fill_state_dict (name-seeded)."""
    from tests.weights import fill_state_dict, surface_inputs
    ref_loader.install()
    import backbones as rb
    import decoders as rd
    x, x2, feat, tg_pad, ln = surface_inputs()
    tx = torch.from_numpy(x)
    out = {}
    with torch.no_grad():
        m = fill_state_dict(rb.resnet18(pretrained=False), "r18.").eval()
        for i, f in enumerate(m(tx)):
            out["r18.%d" % i] = f.numpy()
        m = fill_state_dict(rb.resnet50dilated_ppm(), "ppm.").eval()
        out["ppm"] = m(tx).numpy()
        m = fill_state_dict(rb.Resnet50FPN(resnet_pretrained=False), "fpn50.").eval()
        out["fpn50"] = m(tx).numpy()
    # training-mode trunk (batch statistics) with a gradient norm per stage
    m = fill_state_dict(rb.Resnet18FPN(resnet_pretrained=False), "fpn18.").train()
    y = m(torch.from_numpy(x2))
    y.square().mean().backward()
    out["fpn18.train"] = y.detach().numpy()
    for k in ("bottom_up.conv1.weight", "bottom_up.layer3.0.downsample.0.weight", "top_down.merge_layer.weight"):
        out["fpn18.gnorm." + k] = np.float64(dict(m.named_parameters())[k].grad.double().norm().item())

    tf, tt, tl = torch.from_numpy(feat), torch.from_numpy(tg_pad), torch.from_numpy(ln)
    att = fill_state_dict(rd.AttentionDecoder(256, gt_as_output=True), "attn.").train()
    loss, amap = att(tf, targets=tt, lengths=tl)
    loss.sum().backward()
    out["attn.loss"] = loss.detach().numpy()
    out["attn.map"] = amap.detach().numpy()
    for k in ("encode.0.0.weight", "decoder.attn.attn.weight", "decoder.attn.v", "decoder.rnn.weight_hh",
              "decoder.embedding.weight", "onehot_embedding_x.weight"):
        out["attn.gnorm." + k] = np.float64(dict(att.named_parameters())[k].grad.double().norm().item())
    with torch.no_grad():
        out["attn.eval"] = att.eval()(tf).numpy()
    ctc = fill_state_dict(rd.CTCDecoder(256), "ctc1d.")
    with torch.no_grad():                                     # eval first: pristine BN running statistics
        out["ctc1d.eval"] = ctc.eval()(tf, train=False).numpy()
    loss, lp = ctc.train()(tf, targets=tt, lengths=tl, train=True)
    loss.backward()
    out["ctc1d.loss"] = np.float64(loss.item())
    out["ctc1d.log_probs"] = lp.detach().numpy()
    for k in ("encode.0.0.weight", "pred_conv.weight", "pred_conv.bias"):
        out["ctc1d.gnorm." + k] = np.float64(dict(ctc.named_parameters())[k].grad.double().norm().item())
    np.savez_compressed(os.path.join(GOLD, "surfaces_ref.npz"), **out)
    print("surfaces", {k: getattr(v, "shape", v) for k, v in out.items()})


def make_head():
    """2D-CTC head epilogue (decoders/ctc_decoder2d.py:37-45): run the UNMODIFIED reference module on CPU with its
    `ctc_loss` replaced by a fixed linear functional of `pred`, capture the two conv branches' raw outputs with
    forward hooks, and record pred plus the gradients that reach those raw outputs."""
    import types
    from tests.weights import fill_state_dict
    ref_loader.install()
    ops_stub = types.ModuleType("ops")
    ops_stub.ctc_loss_2d = None
    saved = sys.modules.get("ops")
    sys.modules["ops"] = ops_stub
    try:
        import decoders as rd
        dec = fill_state_dict(rd.CTCDecoder2D(16, inner_channels=8), "d2.").train()
    finally:
        if saved is not None:
            sys.modules["ops"] = saved
        else:
            del sys.modules["ops"]
    rng = np.random.RandomState(21)
    feat = torch.from_numpy((rng.standard_normal((5, 16, 8, 32)) * 3.0).astype(np.float32))
    weight = torch.from_numpy(rng.standard_normal((32, 8, 5, 38)).astype(np.float32))
    lengths = torch.tensor([3, 1, 4, 2, 5])
    captured = {}

    def grab(name):
        def hook(module, inputs, output):
            output.retain_grad()
            captured[name] = output
        return hook
    dec.pred_mask[2].register_forward_hook(grab("mask_logits"))
    dec.pred_classify[2].register_forward_hook(grab("cls_logits"))
    dec.ctc_loss = lambda pred, *a: (pred * weight).sum(dim=(0, 1, 3))
    out = {}
    # case "a": `saved_tiny` as fill_state_dict left it (a large value: the clamp and its zero gradient hit ~half the
    # entries); "b": the real tiny = finfo(float32).tiny, ordinary logits; "c": real tiny, 1x1 convs scaled x25 so that
    # part of mask*classify underflows below tiny
    real_tiny = float(torch.finfo(torch.float32).tiny)
    for tag, tiny, gain in (("a", None, 1.0), ("b", real_tiny, 1.0), ("c", real_tiny, 25.0)):
        with torch.no_grad():
            if tiny is not None:
                dec.saved_tiny.fill_(tiny)
            dec.pred_mask[2].weight.mul_(gain)
            dec.pred_classify[2].weight.mul_(gain)
        dec.zero_grad()
        loss, pred = dec(feat, targets=torch.zeros(5, 32), lengths=lengths, train=True)
        loss.sum().backward()
        dlp = (weight / lengths.float().view(1, 1, -1, 1)).contiguous()      # the upstream gradient that reached pred
        out.update({tag + ".tiny": np.float32(dec.saved_tiny.item()),
                    tag + ".mask_logits": captured["mask_logits"].detach().numpy(),
                    tag + ".cls_logits": captured["cls_logits"].detach().numpy(), tag + ".pred": pred.detach().numpy(),
                    tag + ".grad_pred": dlp.numpy(), tag + ".grad_mask_logits": captured["mask_logits"].grad.numpy(),
                    tag + ".grad_cls_logits": captured["cls_logits"].grad.numpy()})
        print("head", tag, tuple(pred.shape), "tiny", dec.saved_tiny.item(), "clamped fraction",
              float((pred <= float(np.log(dec.saved_tiny.item())) + 1e-6).float().mean()))
    np.savez_compressed(os.path.join(GOLD, "ctc2d_head_ref.npz"), **out)


def make_input():
    """Recognition input step (crnn.yaml processes): run the UNMODIFIED reference ResizeImage (modes resize and pad),
    NormalizeImage and MakeRecognitionLabel on CPU (cv2 4.x from this image) and record their outputs."""
    ref_loader.install()
    from data.processes.resize_image import ResizeImage
    from data.processes.normalize_image import NormalizeImage
    from data.processes.make_recognition_label import MakeRecognitionLabel
    from tests.input_cases import MODES, input_cases
    images, texts = input_cases()
    out = {}
    for mode, size in MODES.items():
        rz = ResizeImage(mode=mode, image_size=list(size))
        nm = NormalizeImage()
        batch = []
        for im in images:
            d = {"image": im.astype("float32")}                     # data/lmdb_dataset.py:87
            d = nm.process(rz.process(d))
            batch.append(d["image"].numpy())
        out["image." + mode] = np.stack(batch)
    mk = MakeRecognitionLabel()
    labels, lengths = [], []
    for t in texts:
        d = mk.process({"gt": t})
        labels.append(np.asarray(d["label"], np.int32))
        lengths.append(int(d["length"]))
    out["labels"] = np.stack(labels)
    out["lengths"] = np.asarray(lengths, np.int32)
    np.savez_compressed(os.path.join(GOLD, "input_ref.npz"), **out)
    print("input", {k: v.shape for k, v in out.items()})


def _keys(m):
    return [[k, list(v.shape)] for k, v in m.state_dict().items()]


def make_crnn_port():
    """Outputs of the reference crnn_backbone + CRNNDecoder (train: loss and log-probs; eval: probabilities) on the batch
    tests/test_oracle_crnn.py feeds the oracle port, and the two modules' state-dict keys."""
    from tests.weights import crnn_batch, fill_state_dict
    ref_loader.install()
    import backbones as rb
    import decoders as rd
    rbb = fill_state_dict(rb.crnn_backbone(), "bb.")
    rdec = fill_state_dict(rd.CRNNDecoder(in_channels=512, inner_channels=256), "dec.")
    torch.set_num_threads(1)                                      # the summation order the test reproduces
    tx, tl, tn = (torch.from_numpy(a) for a in crnn_batch(3, 2, 100, 8, 26))
    loss, pred = rdec(rbb.train()(tx), targets=tl, lengths=tn, train=True)
    with torch.no_grad():
        prob = rdec.eval()(rbb.eval()(tx), train=False)
    np.savez_compressed(os.path.join(GOLD, "crnn_ref_port.npz"), loss=loss.detach().numpy(), log_probs=pred.detach().numpy(),
                        eval_prob=prob.numpy(), bb_keys=np.array(list(rbb.state_dict())),
                        dec_keys=np.array(list(rdec.state_dict())))
    print("crnn_port loss", loss.detach().numpy())


def make_state_dicts():
    """State-dict keys and shapes of the reference's trunk / head modules (tests/test_surfaces_cpu.py) and of the models its three
    recognition yamls build through its own structure/model.py (tests/test_boundary_yaml_cpu.py)."""
    import gzip
    import json
    import types
    import yaml
    ref_loader.install()
    for name in ("assets.ops.dcn.deform_conv_cuda", "assets.ops.dcn.deform_pool_cuda", "ops.ctc_2d.ctc_2d_csrc"):
        sys.modules.setdefault(name, types.ModuleType(name))     # native extensions: only the module definitions are needed
    import backbones as rb
    import decoders as rd
    import structure.model as smodel
    import concern.charsets as charsets
    import assets.ops.dcn.modules.deform_pool as rpool
    out = {"modules": {
        "resnet34": _keys(rb.resnet34(pretrained=False)), "resnet101": _keys(rb.resnet101(pretrained=False)),
        "Resnet34FPN": _keys(rb.Resnet34FPN(resnet_pretrained=False)),
        "resnet50dilated_ppm": _keys(rb.resnet50dilated_ppm(inner_channels=128)),
        "AttentionDecoder": _keys(rd.AttentionDecoder(64, inner_channels=128, max_size=16, height=2)),
        "CTCDecoder": _keys(rd.CTCDecoder(64, inner_channels=96)), "EASTDecoder": _keys(rd.EASTDecoder(channels=64)),
        "deformable_resnet50": _keys(rb.deformable_resnet50(pretrained=False)),
        "ResNet_v1_dcn": _keys(rb.resnet.ResNet(rb.resnet.BasicBlock, [1, 1, 1, 1], dcn=dict(modulated=False, deformable_groups=2))),
        "DeformRoIPoolingPack": _keys(rpool.DeformRoIPoolingPack(0.5, 3, 8, False, trans_std=0.1, deform_fc_channels=32)),
        "ModulatedDeformRoIPoolingPack": _keys(rpool.ModulatedDeformRoIPoolingPack(0.5, 3, 8, False, trans_std=0.1,
                                                                                   deform_fc_channels=32))}}
    out["resnet50dilated_ppm_conv_geometry"] = [[n, list(c.stride), list(c.dilation), list(c.padding)]
                                                for n, c in rb.resnet50dilated_ppm().named_modules()
                                                if isinstance(c, torch.nn.Conv2d)]
    ydir = os.path.join(ref_loader.REF, "experiments", "recognition")
    base = yaml.safe_load(open(os.path.join(ydir, "community-base.yaml")))
    cs_def = [d for d in base["define"] if d["name"] == "charset"][0]
    charset = getattr(charsets, cs_def["class"])()
    out["charset"] = {"class": cs_def["class"], "len": len(charset)}
    out["yamls"] = {}
    for y in ("crnn.yaml", "res50-ppm-2d-ctc.yaml", "fpn50-attention-decoder.yaml"):
        conf = yaml.safe_load(open(os.path.join(ydir, y)))
        builder = [d for d in conf["define"] if d["name"] == "BasicStructure"][0]["builder"]
        args = json.loads(json.dumps(builder["model_args"]))
        if "resnet" in args["backbone"].lower():
            args.setdefault("backbone_args", {})["resnet_pretrained"] = False      # no network for the torchvision checkpoint
        built = json.loads(json.dumps(args))
        for k, v in list(built.get("decoder_args", {}).items()):
            if v == "^charset":
                built["decoder_args"][k] = charset
        model = getattr(smodel, builder["model"])(built, torch.device("cpu"))      # structure/model.py:160-166 -> BasicModel :16-24
        state = model.state_dict()
        assert all(k.startswith("model.module.") for k in state)                  # nn.DataParallel(BasicModel) on one device
        out["yamls"][y] = {"model": builder["model"], "model_args": args,
                           "state": {k[len("model.module."):]: list(v.shape) for k, v in state.items()},
                           "n_params": sum(p.numel() for p in model.parameters())}
    with gzip.open(os.path.join(GOLD, "state_dicts_ref.json.gz"), "wt") as f:
        json.dump(out, f, sort_keys=True)
    print("state_dicts", sorted(out["modules"]), sorted(out["yamls"]))


def make_east():
    """decoders/east.py on CPU, train and eval branches, weights from tests.weights.fill_state_dict (name-seeded)."""
    ref_loader.install()
    import decoders as rd
    from tests.weights import east_inputs, fill_state_dict
    r = fill_state_dict(rd.EASTDecoder(channels=32), "east.").train()
    torch.set_num_threads(1)                                      # the summation order the test reproduces
    x, label = east_inputs()
    loss, pred, metrics = r(x, label, None, True)
    out = {"loss": loss.detach().numpy()}
    out.update({"pred." + k: v.detach().numpy() for k, v in pred.items()})
    out.update({"metrics." + k: v.detach().numpy() for k, v in metrics.items()})
    with torch.no_grad():
        out.update({"eval." + k: v.numpy() for k, v in r.eval()(x, label, None, False).items()})
    np.savez_compressed(os.path.join(GOLD, "east_ref.npz"), **out)
    print("east", {k: v.shape for k, v in out.items()})


def make_ref_kernels():
    """The reference's own CUDA ops (oracle/_ref/*.so from oracle/build_ref.py), run on a GPU on the seeded inputs of
    tests/test_ref_kernels_gpu.py; records their outputs in the form that test compares against."""
    from oracle import build_ref
    from tests import test_ref_kernels_gpu as t
    from tests.deform_pool_cases import CASES as POOL_CASES, make as pool_make
    mods = {n: build_ref.load(n) for n in ("ref_ctc2d", "ref_deform_conv", "ref_deform_pool")}
    if None in mods.values() or not torch.cuda.is_available():
        raise RuntimeError("needs a CUDA device and oracle/_ref/*.so (python -m oracle.build_ref)")
    dev = torch.device("cuda:0")
    dv = lambda *arrs: [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in arrs]  # noqa: E731
    out = {}
    ref = mods["ref_ctc2d"]
    for case in t.CTC_CASES:
        for tag, dtype in t.CTC_DTYPES.items():
            if t.ctc_skip_reason(case, dtype):
                continue
            key = "ctc.%d.%s" % (case[0], tag)
            d_lp, d_tg, d_il, d_tl, d_go = dv(*t.ctc_inputs(case, dtype))
            nll, la = ref.ctc2d_forward(d_lp, d_tg, d_il, d_tl, 0, 0.0)
            gr = ref.ctc2d_backward(d_go, d_lp, d_tg, d_il, d_tl, nll, la, 0)
            out[key + ".nll"] = nll.cpu().numpy()
            t.record(out, key + ".log_alpha", la.cpu().numpy())
            t.record(out, key + ".grad", gr.cpu().numpy())
    ref = mods["ref_deform_conv"]
    for i, case in enumerate(t.DCN_CASES):
        B, C, H, W, Cout, k, s, p, d, group, dg, with_bias, big = case
        x, w, b, off, m, go, Ho, Wo = t._dcn_inputs(11, B, C, H, W, Cout, k, s, p, d, group, dg, big)
        tx, tw, tb, toff, tm, tgo = dv(x, w, b, off, m, go)
        e = lambda: tx.new_empty(0)  # noqa: E731
        r_out = tx.new_empty(B, Cout, Ho, Wo)
        ref.modulated_deform_conv_cuda_forward(tx, tw, tb, e(), toff, tm, r_out, e(), k, k, s, s, p, p, d, d, group, dg, with_bias)
        grads = [torch.zeros_like(v) for v in (tx, tw, tb, toff, tm)]
        ref.modulated_deform_conv_cuda_backward(tx, tw, tb, e(), toff, tm, e(), *grads, tgo, k, k, s, s, p, p, d, d, group, dg,
                                                with_bias)
        key = "dcn2.%d." % i
        for name, v in zip(("output", "grad_input", "grad_weight", "grad_bias", "grad_offset", "grad_mask"), [r_out] + grads):
            t.record(out, key + name, v.cpu().numpy())
        if big:
            out[key + "grad_offset_tail_max_abs"] = np.float64(grads[3].view(B, -1)[:, 2 * k * k * dg * Ho * Wo:].abs().max())
    for name, case in t.DCNV1_CASES.items():
        B, C, H, W, Cout, k, s, p, d, group, dg = case
        x, w, _, off, _, go, Ho, Wo = t._dcn_inputs(12, B, C, H, W, Cout, k, s, p, d, group, dg, False)
        tx, tw, toff, tgo = dv(x, w, off, go)
        e = lambda: tx.new_empty(0)  # noqa: E731
        # im2col_step = B, as functions/deform_conv.py:43 picks for B <= 64.  (The reference's forward re-views `columns` inside
        # its batch loop, deform_conv_cuda.cpp:225, so more than one loop iteration cannot work at all.)
        r_out = tx.new_empty(B, Cout, Ho, Wo)
        ref.deform_conv_forward_cuda(tx, tw, toff, r_out, e(), e(), k, k, s, s, p, p, d, d, group, dg, B)
        r_gi, r_goff, r_gw = torch.zeros_like(tx), torch.zeros_like(toff), torch.zeros_like(tw)
        ref.deform_conv_backward_input_cuda(tx, toff, tgo, r_gi, r_goff, tw, e(), k, k, s, s, p, p, d, d, group, dg, B)
        # backward_parameters does zeros_like(transposed view).view(...) (deform_conv_cuda.cpp:423-430), which only works with
        # today's stride-preserving zeros_like when the transposed dimension has size 1: one sample per call, accumulating
        # into gradWeight exactly as the op is specified to do
        for bi in range(B):
            ref.deform_conv_backward_parameters_cuda(tx[bi:bi + 1], toff[bi:bi + 1], tgo[bi:bi + 1], r_gw, e(), e(), k, k, s, s, p,
                                                     p, d, d, group, dg, 1.0, 1)
        for key, v in (("output", r_out), ("grad_input", r_gi), ("grad_offset", r_goff), ("grad_weight", r_gw)):
            t.record(out, "dcn1.%s.%s" % (name, key), v.cpu().numpy())
    ref = mods["ref_deform_pool"]
    for name in sorted(POOL_CASES):
        data, rois, trans, a = pool_make(name)
        d, r = dv(data.astype(np.float32), rois.astype(np.float32))
        tr = dv(trans.astype(np.float32))[0] if trans is not None else d.new_empty(0)
        n, od, P = rois.shape[0], a["output_dim"], a["pooled"]
        r_out, r_cnt = d.new_zeros(n, od, P, P), d.new_zeros(n, od, P, P)
        ref.deform_psroi_pooling_cuda_forward(d, r, tr, r_out, r_cnt, *t.pool_args(a))
        r_gin, r_gtr = torch.zeros_like(d), torch.zeros_like(tr)
        ref.deform_psroi_pooling_cuda_backward(dv(t.pool_grad_out(n, od, P))[0], d, r, tr, r_cnt, r_gin, r_gtr, *t.pool_args(a))
        for key, v in (("out", r_out), ("count", r_cnt), ("grad_input", r_gin), ("grad_trans", r_gtr)):
            out["pool.%s.%s" % (name, key)] = v.cpu().numpy()
    torch.cuda.synchronize()
    import hashlib
    import json
    import subprocess
    driver = subprocess.run(["nvidia-smi", "--query-gpu=driver_version", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True).stdout.strip()
    out["provenance"] = np.array(json.dumps({
        "gpu": torch.cuda.get_device_name(0), "driver": driver, "torch": torch.__version__, "cuda": torch.version.cuda,
        "reference_binaries_sha256": {n: hashlib.sha256(open(build_ref.so_path(n), "rb").read()).hexdigest() for n in mods}},
        sort_keys=True))
    np.savez_compressed(os.path.join(GOLD, "ref_kernels.npz"), **out)
    print("ref_kernels", len(out), "arrays")


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    which = sys.argv[1:] or ["ctc2d"]
    if "ctc2d" in which:
        make_ctc2d()
    if "crnn" in which:
        make_crnn()
    if "surfaces" in which:
        make_surfaces()
    if "head" in which:
        make_head()
    if "input" in which:
        make_input()
    if "crnn_port" in which:
        make_crnn_port()
    if "state_dicts" in which:
        make_state_dicts()
    if "east" in which:
        make_east()
    if "ref_kernels" in which:
        make_ref_kernels()
