"""Record tests/golden/db_ref.npz from the UNMODIFIED reference DB detector (decoders/seg_detector.py,
decoders/seg_detector_loss.py) on the CPU.

Run:  python -m oracle.make_golden_db            (from the repo root; needs the reference checkout, see oracle/ref_loader.py)

Records:
  head.*      SegDetector(adaptive=True, in_channels=[256,512,1024,2048], k=50) outputs, name-seeded weights (tests/weights.py),
              on seeded features of a 32x32 input, train (batch statistics) and eval
  loss<i>.*   the inputs, loss, metrics and the gradients of the loss w.r.t. binary / thresh / thresh_binary of L1BalanceCELoss in
              float64 for seeded batches (oracle/db_port.py db_batch), N = 1, 2, 3
  keys        state-dict keys and shapes of that SegDetector and of the model experiments/seg_detector/seg_detector_db.yaml builds
"""
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import db_port, ref_loader  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
HEAD_ARGS = dict(adaptive=True, in_channels=[256, 512, 1024, 2048], k=50)
LOSS_CASES = [(1, 1, 24, 32), (2, 2, 20, 28), (3, 3, 17, 23)]       # seed, N, H, W


def head_features(seed=5, n=2, hw=32):
    rng = np.random.RandomState(seed)
    return [torch.from_numpy(rng.standard_normal((n, c, hw // s, hw // s)).astype(np.float32))
            for c, s in ((256, 4), (512, 8), (1024, 16), (2048, 32))]


def main():
    ref_loader.install()
    for name in ("assets.ops.dcn.deform_conv_cuda", "assets.ops.dcn.deform_pool_cuda"):
        sys.modules.setdefault(name, types.ModuleType(name))     # native extensions: only the module definitions are needed
    import structure.model as smodel
    from decoders.seg_detector import SegDetector
    from decoders.seg_detector_loss import SegDetectorLossBuilder
    from tests.weights import fill_state_dict
    import yaml
    torch.set_num_threads(1)                                      # the summation order the test reproduces
    out = {}
    head = fill_state_dict(SegDetector(**HEAD_ARGS), "db.").train()
    feats = head_features()
    with torch.no_grad():
        for mode in ("train", "eval"):
            res = head.train(mode == "train")(feats)
            out.update({"head.%s.%s" % (mode, k): v.numpy() for k, v in res.items()})
    crit = SegDetectorLossBuilder("L1BalanceCELoss").build()
    for i, (seed, N, H, W) in enumerate(LOSS_CASES):
        pred, batch = db_port.db_batch(seed, N, H, W, torch.float64)
        pred = {k: v.requires_grad_(True) for k, v in pred.items()}
        loss, metrics = crit(pred, batch)
        grads = torch.autograd.grad(loss, [pred["binary"], pred["thresh"], pred["thresh_binary"]])
        out.update({"loss%d.in.%s" % (i, k): v.detach().numpy() for k, v in list(pred.items()) + list(batch.items())})
        out["loss%d.loss" % i] = loss.detach().numpy()
        out.update({"loss%d.metrics.%s" % (i, k): v.detach().numpy() for k, v in metrics.items()})
        out.update({"loss%d.grad.%s" % (i, k): g.numpy() for k, g in zip(("binary", "thresh", "thresh_binary"), grads)})
        print("db loss case", i, float(loss), {k: float(v) for k, v in metrics.items()})
    conf = yaml.safe_load(open(os.path.join(ref_loader.REF, "experiments", "seg_detector", "seg_detector_db.yaml")))
    exp = [d for d in conf["define"] if d["name"] == "Experiment"][0]
    builder = exp["structure"]["builder"]
    args = json.loads(json.dumps(builder["model_args"]))
    args.setdefault("backbone_args", {})["pretrained"] = False                     # no network for the torchvision checkpoint
    model = getattr(smodel, builder["model"])(args, torch.device("cpu"))           # structure/model.py:126-138
    state = {k[len("model.module."):]: list(v.shape) for k, v in model.state_dict().items() if k.startswith("model.module.")}
    keys = {"SegDetector": [[k, list(v.shape)] for k, v in head.state_dict().items()],
            "yaml": {"model": builder["model"], "model_args": args, "state": state,
                     "n_params": sum(p.numel() for p in model.model.parameters())}}
    out["keys_json"] = np.array(json.dumps(keys, sort_keys=True))
    np.savez_compressed(os.path.join(GOLD, "db_ref.npz"), **out)
    print("db_ref", len(out), "arrays,", len(state), "yaml state entries")


if __name__ == "__main__":
    main()
