"""Deterministic, torch-version-independent parameter values keyed by parameter NAME, so the reference modules
(build container, oracle/make_golden.py) and megreader_b200's modules (GPU box) hold identical weights without
shipping 33 MB state dicts."""
import zlib

import numpy as np
import torch


def fill_state_dict(module, salt=""):
    sd = module.state_dict()
    new = {}
    for name in sorted(sd):
        t = sd[name]
        if not t.is_floating_point():
            new[name] = t.clone()
            continue
        rng = np.random.RandomState(zlib.crc32((salt + name).encode()) & 0x7FFFFFFF)
        shape = tuple(t.shape)
        if name.endswith("running_var"):
            v = 1.0 + 0.1 * np.abs(rng.standard_normal(shape))
        elif name.endswith("running_mean"):
            v = 0.1 * rng.standard_normal(shape)
        elif t.dim() >= 2:
            fan_in = int(np.prod(shape[1:]))
            v = rng.standard_normal(shape) * (1.0 / np.sqrt(fan_in))
        elif name.endswith("weight"):          # BatchNorm weight
            v = 1.0 + 0.1 * rng.standard_normal(shape)
        else:                                   # biases
            v = 0.05 * rng.standard_normal(shape)
        new[name] = torch.from_numpy(np.asarray(v, dtype=np.float32)).reshape(shape).to(t.dtype)
    module.load_state_dict(new)
    return module


def crnn_batch(seed, N, W, L_max, T, n_classes=38, S=32):
    """SURVEY.md §8d synthetic lines: x = randn(N,3,32,W) (one gray channel replicated x3, D2); labels U{2..37},
    length U{1..L_max} with 2*length+1 <= T, blank-padded to S=32 int32 like concern/charsets.py:52-58."""
    rng = np.random.RandomState(seed)
    gray = rng.standard_normal((N, 1, 32, W)).astype(np.float32)
    x = np.repeat(gray, 3, axis=1)
    L_max = min(L_max, (T - 1) // 2)
    lengths = rng.randint(1, L_max + 1, size=N).astype(np.int64)
    labels = np.zeros((N, S), np.int32)
    for b in range(N):
        labels[b, :lengths[b]] = rng.randint(2, n_classes, size=lengths[b])
    return x, labels, lengths


def surface_inputs():
    """Seeded inputs of tests/golden/surfaces_ref.npz (regenerated on both sides instead of stored)."""
    rng = np.random.RandomState(11)
    x = rng.standard_normal((1, 3, 32, 64)).astype(np.float32)
    x2 = rng.standard_normal((2, 3, 32, 64)).astype(np.float32)
    feat = (rng.standard_normal((3, 256, 16, 64)) * 0.5).astype(np.float32)
    lengths = np.array([5, 9, 31], np.int64)
    targets = rng.randint(2, 38, size=(3, 32)).astype(np.int64)
    for b in range(3):
        targets[b, lengths[b]:] = 0
    return x, x2, feat, targets, lengths


def east_inputs():
    """Seeded inputs of tests/golden/east_ref.npz: a 32-channel feature map and EAST labels at 4x its resolution."""
    rng = np.random.RandomState(0)
    x = rng.standard_normal((2, 32, 3, 5)).astype(np.float32)
    label = {"heatmap": (rng.random_sample((2, 1, 12, 20)) > 0.7).astype(np.float32),
             "heatmap_weight": rng.random_sample((2, 1, 12, 20)).astype(np.float32),
             "densebox": (rng.standard_normal((2, 8, 12, 20)) * 50).astype(np.float32),
             "densebox_weight": rng.random_sample((2, 8, 12, 20)).astype(np.float32)}
    return torch.from_numpy(x), {k: torch.from_numpy(v) for k, v in label.items()}
