"""CPU: the reference's three recognition yamls build UNCHANGED on megreader_b200's surfaces.

`python -m oracle.make_golden state_dicts` built each yaml's model with the reference's own structure/model.py
(SequenceRecognitionModel :160-181 -> BasicModel :16-24) and concern/charsets.py on the reference's modules, and recorded its
`model_args`, state dict (names and shapes: what checkpoints hold) and parameter count in tests/golden/state_dicts_ref.json.gz.
The same `model_args`, resolved through `getattr(backbones, name)` / `getattr(decoders, name)` (structure/model.py:20-21) to
megreader_b200/refapi, must give the same state dict."""
import gzip
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_yamls_build_on_refapi_with_identical_state_dicts():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "boundary_probe.py")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    ours = json.loads(r.stdout.strip().splitlines()[-1])
    with gzip.open(os.path.join(ROOT, "tests", "golden", "state_dicts_ref.json.gz"), "rt") as f:
        ref = json.load(f)
    assert "refapi" in ours["backbones_file"] and "refapi" in ours["decoders_file"]
    assert ours["charset_len"] == ref["charset"]["len"]
    assert set(ours["models"]) == {"crnn.yaml", "res50-ppm-2d-ctc.yaml", "fpn50-attention-decoder.yaml"} == set(ref["yamls"])
    for y, m in ours["models"].items():
        r = ref["yamls"][y]
        assert (m["model"], m["backbone"], m["decoder"]) == (r["model"], r["model_args"]["backbone"], r["model_args"]["decoder"])
        assert m["n_params"] == r["n_params"], y
        assert m["state"] == r["state"], (y, sorted(set(m["state"]) ^ set(r["state"]))[:10])
