"""CPU: the CRNN oracle port (oracle/crnn_port.py) equals the UNMODIFIED reference modules bit-for-bit, and reproduces the
committed golden vectors anywhere."""
import os

import numpy as np
import torch

from oracle import crnn_port
from tests.weights import crnn_batch, fill_state_dict

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _port():
    bb = fill_state_dict(crnn_port.CRNNBackbonePort(), "bb.")
    dec = fill_state_dict(crnn_port.CRNNDecoderPort(), "dec.")
    return bb, dec


def test_port_reproduces_golden():
    g = np.load(os.path.join(GOLD, "crnn_ref_cfg1.npz"))
    bb, dec = _port()
    torch.set_num_threads(1)
    x = torch.from_numpy(np.repeat(g["x"], 3, axis=1))
    loss, pred = dec(bb.train()(x), torch.from_numpy(g["labels"]), torch.from_numpy(g["lengths"]), train=True)
    np.testing.assert_allclose(loss.item(), float(g["loss"]), rtol=1e-5)
    np.testing.assert_allclose(pred.detach().numpy(), g["log_probs"], rtol=1e-4, atol=1e-5)


def test_port_equals_unmodified_reference():
    """The unmodified reference modules' train and eval outputs on this batch, recorded by `python -m oracle.make_golden
    crnn_port` into tests/golden/crnn_ref_port.npz with one host thread: the port computes them bit for bit."""
    g = np.load(os.path.join(GOLD, "crnn_ref_port.npz"))
    bb, dec = _port()
    torch.set_num_threads(1)
    assert list(bb.state_dict()) == list(g["bb_keys"]) and list(dec.state_dict()) == list(g["dec_keys"])
    x, labels, lengths = crnn_batch(3, 2, 100, 8, 26)
    tx, tl, tn = torch.from_numpy(x), torch.from_numpy(labels), torch.from_numpy(lengths)
    b = dec(bb.train()(tx), tl, tn, train=True)
    assert torch.equal(b[0], torch.from_numpy(g["loss"])) and torch.equal(b[1], torch.from_numpy(g["log_probs"]))
    with torch.no_grad():
        pb = dec.eval()(bb.eval()(tx), train=False)
    assert torch.equal(pb, torch.from_numpy(g["eval_prob"]))
