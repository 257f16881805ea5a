"""Loss of the DB text detector with the reference's surface (decoders/seg_detector_loss.py:7-33 and 157-185): SegDetectorLossBuilder
and L1BalanceCELoss(eps=1e-6, l1_scale=10, bce_scale=5), returning (loss, {'bce_loss', 'thresh_loss', 'l1_loss'}).

    bce  = balanced BCE on `binary`: every positive pixel plus the 3x-as-many hardest negatives, where gt (N,1,H,W) times
           mask (N,H,W) broadcasts to (N,N,H,W) -- every sample's gt is paired with every sample's mask, as in the reference
    dice = 1 - 2 sum(tb g m) / (sum(tb m) + sum(g m) + eps)          on `thresh_binary`
    l1   = sum(|thresh - thresh_map| thresh_mask) / sum(thresh_mask)
    loss = dice + l1_scale l1 + bce_scale bce

On CUDA tensors the whole loss runs on csrc/db_head.cu (megreader_b200/db.py): nothing of size N^2 H W, no host synchronisation,
sums in fp64, exact integer counts, the dice `assert loss <= 1` not evaluated (it would synchronise), and the gradient split
evenly among negatives tied at the selection threshold (torch.topk picks among them in an unspecified order; the loss value is
the same).  On CPU tensors the framework composition below runs."""
import sys

import torch
import torch.nn as nn


class SegDetectorLossBuilder():
    """SegDetectorLossBuilder('L1BalanceCELoss', *args, **kwargs).build() -> the loss module."""

    PROVIDED = ('L1BalanceCELoss',)

    def __init__(self, loss_class, *args, **kwargs):
        self.loss_class = loss_class
        self.loss_args = args
        self.loss_kwargs = kwargs

    def build(self):
        if self.loss_class not in self.PROVIDED:
            raise NotImplementedError("megreader_b200: SegDetector loss %r is not provided; available: %s"
                                      % (self.loss_class, ", ".join(self.PROVIDED)))
        return getattr(sys.modules[__name__], self.loss_class)(*self.loss_args, **self.loss_kwargs)


def _balance_bce(pred, gt, mask, negative_ratio=3.0, eps=1e-6):
    positive = (gt * mask).byte()                    # (N,1,H,W) x (N,H,W) -> (N,N,H,W)
    negative = ((1 - gt) * mask).byte()
    positive_count = int(positive.float().sum())
    negative_count = min(int(negative.float().sum()), int(positive_count * negative_ratio))
    loss = nn.functional.binary_cross_entropy(pred, gt, reduction='none')[:, 0, :, :]
    positive_loss = loss * positive.float()
    negative_loss, _ = torch.topk((loss * negative.float()).view(-1), negative_count)
    return (positive_loss.sum() + negative_loss.sum()) / (positive_count + negative_count + eps)


def _dice(pred, gt, mask, eps):
    pred, gt = pred[:, 0, :, :], gt[:, 0, :, :]
    intersection = (pred * gt * mask).sum()
    union = (pred * mask).sum() + (gt * mask).sum() + eps
    loss = 1 - 2.0 * intersection / union
    assert loss <= 1
    return loss


def _mask_l1(pred, gt, mask):
    return (torch.abs(pred[:, 0] - gt) * mask).sum() / mask.sum()


class L1BalanceCELoss(nn.Module):
    """Balanced cross entropy on `binary`, masked L1 on `thresh`, dice on `thresh_binary`."""

    def __init__(self, eps=1e-6, l1_scale=10, bce_scale=5):
        super().__init__()
        self.eps = eps
        self.l1_scale = l1_scale
        self.bce_scale = bce_scale

    def forward(self, pred, batch):
        if pred['binary'].is_cuda:
            from megreader_b200 import db
            out = db.l1_balance_ce_loss(pred['binary'], pred['thresh'], pred['thresh_binary'], batch['gt'], batch['mask'],
                                        batch['thresh_map'], batch['thresh_mask'], self.eps, self.l1_scale, self.bce_scale)
            return out[0], dict(bce_loss=out[1], thresh_loss=out[2], l1_loss=out[3])
        bce_loss = _balance_bce(pred['binary'], batch['gt'], batch['mask'])
        l1_loss = _mask_l1(pred['thresh'], batch['thresh_map'], batch['thresh_mask'])
        dice_loss = _dice(pred['thresh_binary'], batch['gt'], batch['mask'], self.eps)
        loss = dice_loss + self.l1_scale * l1_loss + bce_loss * self.bce_scale
        return loss, dict(bce_loss=bce_loss, thresh_loss=dice_loss, l1_loss=l1_loss)
