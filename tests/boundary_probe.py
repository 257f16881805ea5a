"""Helper of tests/test_boundary_yaml_cpu.py (run as a subprocess, so that the reference's top-level names stay out of the test
process): build the models of the reference's three recognition yamls from their recorded `model_args`, with `backbones` /
`decoders` / `ops` / `assets` resolved to megreader_b200/refapi, composed as structure/model.py:16-24 BasicModel composes them.
Prints one JSON object."""
import gzip
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import megreader_b200  # noqa: E402
from megreader_b200 import charset as mcharset  # noqa: E402

sys.path.insert(0, os.path.join(os.path.dirname(megreader_b200.__file__), "refapi"))
import torch  # noqa: E402
import backbones  # noqa: E402
import decoders  # noqa: E402


class BasicModel(torch.nn.Module):
    def __init__(self, args):
        super().__init__()
        self.backbone = getattr(backbones, args["backbone"])(**args.get("backbone_args", {}))
        self.decoder = getattr(decoders, args["decoder"])(**args.get("decoder_args", {}))


with gzip.open(os.path.join(ROOT, "tests", "golden", "state_dicts_ref.json.gz"), "rt") as f:
    gold = json.load(f)
charset = getattr(mcharset, gold["charset"]["class"])()
out = {"backbones_file": backbones.__file__, "decoders_file": decoders.__file__, "charset_len": len(charset), "models": {}}
for y, rec in gold["yamls"].items():
    args = json.loads(json.dumps(rec["model_args"]))
    for k, v in list(args.get("decoder_args", {}).items()):
        if v == "^charset":
            args["decoder_args"][k] = charset
    model = BasicModel(args)
    out["models"][y] = {"model": rec["model"], "backbone": args["backbone"], "decoder": args["decoder"],
                        "state": {k: list(v.shape) for k, v in model.state_dict().items()},
                        "n_params": sum(p.numel() for p in model.parameters())}
print(json.dumps(out))
