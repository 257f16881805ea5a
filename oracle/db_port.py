"""Plain-torch restatement of the DB detector's probability maps and L1BalanceCELoss (decoders/seg_detector.py:117-147,
decoders/seg_detector_loss.py:157-185, balance_cross_entropy_loss.py:40-54, dice_loss.py:31-42, l1_loss.py:9-11), written out
literally: the (N,1,H,W) x (N,H,W) -> (N,N,H,W) broadcast of gt and mask, torch.topk over it, host int() counts.  Runs on CPU in
float64 (what the tests pin against tests/golden/db_ref.npz and compare the kernels with) and on the GPU in float32 (the library
arm of bench_db.py).

tie_split=True replaces the topk term by its value written through the threshold tau (the k-th largest entry): the entries
above tau, plus the r = k - #above remainder spread evenly over the T entries equal to tau (r / T each), none when tau = 0.  The
value is the same as topk's; the gradient is the one csrc/db_head.cu defines where topk's choice among ties is unspecified."""
import numpy as np
import torch
import torch.nn as nn


def maps(x_b, x_t, k):
    binary = torch.sigmoid(x_b)
    thresh = torch.sigmoid(x_t)
    thresh_binary = torch.reciprocal(1 + torch.exp(-k * (binary - thresh)))
    return binary, thresh, thresh_binary


def balance_bce(pred, gt, mask, negative_ratio=3.0, eps=1e-6, tie_split=False):
    positive = (gt * mask).byte()
    negative = ((1 - gt) * mask).byte()
    positive_count = int(positive.float().sum())
    negative_count = min(int(negative.float().sum()), int(positive_count * negative_ratio))
    loss = nn.functional.binary_cross_entropy(pred, gt, reduction='none')[:, 0, :, :]
    positive_loss = loss * positive.to(loss.dtype)
    negative_loss = (loss * negative.to(loss.dtype)).view(-1)
    top, _ = torch.topk(negative_loss, negative_count)
    if tie_split and negative_count > 0:
        tau = top[-1].detach()
        above = negative_loss > tau
        tied = negative_loss == tau
        r = negative_count - int(above.sum())
        neg_sum = (negative_loss * above).sum()
        if float(tau) > 0:
            neg_sum = neg_sum + (negative_loss * tied).sum() * (r / float(tied.sum()))
    else:
        neg_sum = top.sum()
    return (positive_loss.sum() + neg_sum) / (positive_count + negative_count + eps)


def dice(pred, gt, mask, eps=1e-6):
    pred, gt = pred[:, 0, :, :], gt[:, 0, :, :]
    intersection = (pred * gt * mask).sum()
    union = (pred * mask).sum() + (gt * mask).sum() + eps
    return 1 - 2.0 * intersection / union


def mask_l1(pred, gt, mask):
    return (torch.abs(pred[:, 0] - gt) * mask).sum() / mask.sum()


def l1_balance_ce_loss(pred, batch, eps=1e-6, l1_scale=10, bce_scale=5, tie_split=False):
    bce_loss = balance_bce(pred['binary'], batch['gt'], batch['mask'], tie_split=tie_split)
    l1_loss = mask_l1(pred['thresh'], batch['thresh_map'], batch['thresh_mask'])
    dice_loss = dice(pred['thresh_binary'], batch['gt'], batch['mask'], eps)
    loss = dice_loss + l1_scale * l1_loss + bce_loss * bce_scale
    return loss, dict(bce_loss=bce_loss, thresh_loss=dice_loss, l1_loss=l1_loss)


def db_batch(seed, N, H, W, dtype=torch.float32):
    """Seeded predictions and labels of the loss: binary / thresh / thresh_binary from random logits (k = 50), gt = rectangles of
    text, mask = 1 outside a few ignore rectangles, thresh_map in [0.3, 0.7] on a band around the text, thresh_mask = that band."""
    rng = np.random.RandomState(seed)
    xb = rng.standard_normal((N, 1, H, W)) * 2.0
    xt = rng.standard_normal((N, 1, H, W))
    gt = np.zeros((N, 1, H, W))
    mask = np.ones((N, H, W))
    tmap = np.full((N, H, W), 0.3)
    tmask = np.zeros((N, H, W))
    for n in range(N):
        for _ in range(rng.randint(1, 4)):
            h, w = rng.randint(2, max(3, H // 3)), rng.randint(3, max(4, W // 2))
            y, x = rng.randint(0, H - h), rng.randint(0, W - w)
            y0, y1, x0, x1 = max(0, y - 2), min(H, y + h + 2), max(0, x - 2), min(W, x + w + 2)
            tmask[n, y0:y1, x0:x1] = 1
            tmap[n, y0:y1, x0:x1] = 0.3 + 0.4 * rng.random_sample((y1 - y0, x1 - x0))
            gt[n, 0, y:y + h, x:x + w] = 1
        if rng.random_sample() < 0.7:
            h, w = rng.randint(1, max(2, H // 4)), rng.randint(1, max(2, W // 4))
            y, x = rng.randint(0, H - h), rng.randint(0, W - w)
            mask[n, y:y + h, x:x + w] = 0
    b, t, tb = maps(torch.from_numpy(xb), torch.from_numpy(xt), 50)
    pred = {"binary": b, "thresh": t, "thresh_binary": tb}
    batch = {"gt": torch.from_numpy(gt), "mask": torch.from_numpy(mask), "thresh_map": torch.from_numpy(tmap),
             "thresh_mask": torch.from_numpy(tmask)}
    return {k: v.to(dtype) for k, v in pred.items()}, {k: v.to(dtype) for k, v in batch.items()}
