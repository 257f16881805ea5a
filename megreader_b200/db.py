"""DB text detector (differentiable binarization): SegDetector's probability maps and L1BalanceCELoss on the kernels of
csrc/db_head.cu.  CUDA only, through the C-ABI; no CPU fallback.

    b, t, tb = maps(x_b, x_t, k)                                  # sigmoid, sigmoid, 1 / (1 + exp(-k (b - t)))
    out = l1_balance_ce_loss(b, t, tb, gt, mask, thresh_map, thresh_mask)
    loss, bce_loss, thresh_loss, l1_loss = out[0], out[1], out[2], out[3]

The loss pairs every sample's gt with every sample's mask exactly as the reference's broadcast does
(decoders/balance_cross_entropy_loss.py:40-54) without forming anything of size N^2 H W, and it never synchronises
with the host, so a training step that uses it can be captured in a CUDA graph."""
import torch
from torch.autograd import Function

from . import _lib

NEGATIVE_RATIO = 3.0      # BalanceCrossEntropyLoss() defaults, as L1BalanceCELoss builds it
BCE_EPS = 1e-6


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check(name, x, shape, device):
    if not x.is_cuda:
        raise NotImplementedError("megreader_b200.db: %s must be a CUDA tensor (no CPU fallback)" % name)
    if x.dtype != torch.float32:
        raise TypeError("megreader_b200.db: %s must be float32, got %s" % (name, x.dtype))
    if tuple(x.shape) != tuple(shape):
        raise ValueError("megreader_b200.db: %s has shape %s, expected %s" % (name, tuple(x.shape), tuple(shape)))
    if not x.is_contiguous():
        raise ValueError("megreader_b200.db: %s must be contiguous" % name)
    if x.device != device:
        raise ValueError("megreader_b200.db: %s is on %s, expected %s" % (name, x.device, device))


def _ptr(x):
    return x.data_ptr() if x is not None else None


class MapsFunction(Function):
    """(x_b, x_t) logits of the last transposed convolutions of `binarize` / `thresh` -> (binary, thresh, thresh_binary)."""

    @staticmethod
    def forward(ctx, x_b, x_t, k):
        _check("x_b", x_b, x_b.shape, x_b.device)
        _check("x_t", x_t, x_b.shape, x_b.device)
        b, t, tb = torch.empty_like(x_b), torch.empty_like(x_b), torch.empty_like(x_b)
        with torch.cuda.device(x_b.device):
            _lib.check(_lib.lib().mr_db_maps_fwd_f32(x_b.data_ptr(), x_t.data_ptr(), x_b.numel(), float(k), b.data_ptr(),
                                                     t.data_ptr(), tb.data_ptr(), _stream()), "db_maps_fwd")
        ctx.save_for_backward(b, t, tb)
        ctx.k = float(k)
        return b, t, tb

    @staticmethod
    def backward(ctx, gb, gt, gtb):
        b, t, tb = ctx.saved_tensors
        gb, gt, gtb = (g.contiguous().float() if g is not None else None for g in (gb, gt, gtb))
        gxb, gxt = torch.empty_like(b), torch.empty_like(b)
        with torch.cuda.device(b.device):
            _lib.check(_lib.lib().mr_db_maps_bwd_f32(_ptr(gb), _ptr(gt), _ptr(gtb), b.data_ptr(), t.data_ptr(), tb.data_ptr(),
                                                     b.numel(), ctx.k, gxb.data_ptr(), gxt.data_ptr(), _stream()), "db_maps_bwd")
        return gxb, gxt, None


def maps(x_b, x_t, k):
    return MapsFunction.apply(x_b, x_t, k)


def loss_workspace_bytes(N, HW):
    return int(_lib.lib().mr_db_loss_workspace_bytes(N, HW))


class L1BalanceCELossFunction(Function):
    """(binary, thresh, thresh_binary (N,1,H,W); gt (N,1,H,W); mask, thresh_map, thresh_mask (N,H,W)) ->
    out [4] = (loss, bce_loss, thresh_loss, l1_loss); differentiable in binary, thresh and thresh_binary."""

    @staticmethod
    def forward(ctx, b, t, tb, gt, mask, thresh_map, thresh_mask, eps, l1_scale, bce_scale):
        if b.dim() != 4 or b.shape[1] != 1:
            raise ValueError("megreader_b200.db: binary must be (N,1,H,W), got %s" % (tuple(b.shape),))
        N, _, H, W = b.shape
        dev = b.device
        for name, x, shape in (("binary", b, b.shape), ("thresh", t, b.shape), ("thresh_binary", tb, b.shape),
                               ("gt", gt, b.shape), ("mask", mask, (N, H, W)), ("thresh_map", thresh_map, (N, H, W)),
                               ("thresh_mask", thresh_mask, (N, H, W))):
            _check(name, x, shape, dev)
        ws = torch.empty(loss_workspace_bytes(N, H * W), dtype=torch.uint8, device=dev)
        out = torch.empty(4, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().mr_db_loss_fwd_f32(
                b.data_ptr(), t.data_ptr(), tb.data_ptr(), gt.data_ptr(), mask.data_ptr(), thresh_map.data_ptr(),
                thresh_mask.data_ptr(), N, H * W, float(eps), float(l1_scale), float(bce_scale), NEGATIVE_RATIO, BCE_EPS,
                ws.data_ptr(), ws.numel(), out.data_ptr(), _stream()), "db_loss_fwd")
        ctx.save_for_backward(b, t, gt, mask, thresh_map, thresh_mask, ws)
        ctx.scales = (float(l1_scale), float(bce_scale))
        return out

    @staticmethod
    def backward(ctx, gout):
        b, t, gt, mask, thresh_map, thresh_mask, ws = ctx.saved_tensors
        N, _, H, W = b.shape
        gout = gout.contiguous().float()
        gb, gtt, gtb = torch.empty_like(b), torch.empty_like(b), torch.empty_like(b)
        with torch.cuda.device(b.device):
            _lib.check(_lib.lib().mr_db_loss_bwd_f32(
                gout.data_ptr(), b.data_ptr(), t.data_ptr(), gt.data_ptr(), mask.data_ptr(), thresh_map.data_ptr(),
                thresh_mask.data_ptr(), N, H * W, ctx.scales[0], ctx.scales[1], ws.data_ptr(), ws.numel(), gb.data_ptr(),
                gtt.data_ptr(), gtb.data_ptr(), _stream()), "db_loss_bwd")
        return gb, gtt, gtb, None, None, None, None, None, None, None


def l1_balance_ce_loss(binary, thresh, thresh_binary, gt, mask, thresh_map, thresh_mask, eps=1e-6, l1_scale=10, bce_scale=5):
    return L1BalanceCELossFunction.apply(binary, thresh, thresh_binary, gt, mask, thresh_map, thresh_mask, eps, l1_scale,
                                         bce_scale)
