"""Benchmarks of the DB text detector (experiments/seg_detector/seg_detector_db.yaml of the reference) on one GPU.

    python bench_db.py loss [--reps R]     L1BalanceCELoss forward + backward at (N, H, W) = (2, 640, 640) (the yaml's batch of 16
                                           over 8 GPUs) and (16, 640, 640) (the whole batch on one GPU): csrc/db_head.cu against
                                           the literal framework composition (oracle/db_port.py) on the same device
    python bench_db.py step [--steps K]    the training step at 640 x 640, N = 2 and 16: deformable_resnet50 + SegDetector +
                                           L1BalanceCELoss + SGD(momentum 0.9, weight decay 1e-4); engine path (tcgen05 convolutions
                                           in bf16 + the DB kernels, captured in a CUDA graph) against the fp32 modules with the
                                           literal loss, eager (its host syncs rule out capture)
    python bench_db.py                     both

Each result is one JSON line carrying the GPU name and power limit read in the same run.  Nothing is written to the tree."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FWD_BYTES = 28        # per (sample, pixel): read b, t, tb, gt, mask, thresh_map, thresh_mask (7 fp32)
BWD_BYTES = 36        # per (sample, pixel): read b, t, gt, mask, thresh_map, thresh_mask, write 3 gradients (9 fp32)
YAML_HEAD = dict(adaptive=True, in_channels=[256, 512, 1024, 2048], k=50)


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception as e:                     # reported, not guessed
        info["power_limit_w"] = "unavailable (%s)" % type(e).__name__
    return info


def synth_batch(seed, N, H, W, device):
    """Seeded DB labels made on the device: 6-12 rectangles of text per image (~10-20 % of the pixels), two ignore rectangles
    (mask 0), a 4-pixel band around every rectangle where thresh_mask = 1 and thresh_map in [0.3, 0.7] (0.3 elsewhere, as
    MakeBorderMap leaves it), and a normalised image."""
    g = torch.Generator(device=device).manual_seed(seed)
    ys = torch.arange(H, device=device).view(1, 1, H, 1)
    xs = torch.arange(W, device=device).view(1, 1, 1, W)

    def rects(n, hmax, wmax):
        h = (torch.rand(N, n, 1, 1, generator=g, device=device) * (hmax - 8) + 8).long()
        w = (torch.rand(N, n, 1, 1, generator=g, device=device) * (wmax - 16) + 16).long()
        y = (torch.rand(N, n, 1, 1, generator=g, device=device) * (H - h)).long()
        x = (torch.rand(N, n, 1, 1, generator=g, device=device) * (W - w)).long()
        return y, x, h, w

    def inside(y, x, h, w, keep, pad=0):
        return ((ys >= y - pad) & (ys < y + h + pad) & (xs >= x - pad) & (xs < x + w + pad) & keep).any(1)

    y, x, h, w = rects(12, H // 6, W // 2)
    keep = torch.arange(12, device=device).view(1, 12, 1, 1) < torch.randint(6, 13, (N, 1, 1, 1), generator=g, device=device)
    text = inside(y, x, h, w, keep)
    band = inside(y, x, h, w, keep, pad=4) & ~text
    iy, ix, ih, iw = rects(2, H // 10, W // 10)
    mask = (~inside(iy, ix, ih, iw, True)).float()
    thresh_map = torch.where(band, 0.3 + 0.4 * torch.rand(N, H, W, generator=g, device=device), torch.full_like(mask, 0.3))
    batch = {"image": torch.randn(N, 3, H, W, generator=g, device=device), "gt": text.float().unsqueeze(1), "mask": mask,
             "thresh_map": thresh_map, "thresh_mask": band.float()}
    return batch


def loss_inputs(seed, N, H, W, device):
    """Predictions for the loss benchmark: sigmoid maps of random logits, on top of synth_batch's labels."""
    from oracle import db_port
    batch = synth_batch(seed, N, H, W, device)
    g = torch.Generator(device=device).manual_seed(seed + 1)
    b, t, tb = db_port.maps(2 * torch.randn(N, 1, H, W, generator=g, device=device),
                            torch.randn(N, 1, H, W, generator=g, device=device), 50)
    return {"binary": b, "thresh": t, "thresh_binary": tb}, batch


def _timed(fn, reps, flush=None):
    """Mean ms per call from CUDA events, each call after an L2 flush (a 256 MB write) when `flush` is given."""
    total = 0.0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
    return total / reps


def bench_loss(args, emit):
    from megreader_b200 import _lib, db
    from oracle import db_port
    dev = torch.device("cuda:0")
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)     # 256 MB > the 126 MB L2
    for N in (2, 16):
        H = W = 640
        pred, batch = loss_inputs(100 + N, N, H, W, dev)
        leaves = {k: v.detach().clone().requires_grad_(True) for k, v in pred.items()}
        res = {}
        for arm in ("kernels", "library"):
            def run():
                for v in leaves.values():
                    v.grad = None
                if arm == "kernels":
                    out = db.l1_balance_ce_loss(leaves["binary"], leaves["thresh"], leaves["thresh_binary"], batch["gt"],
                                                batch["mask"], batch["thresh_map"], batch["thresh_mask"])
                    loss = out[0]
                else:
                    loss, _ = db_port.l1_balance_ce_loss(leaves, batch)
                loss.backward()
                return loss
            for _ in range(3):
                run()
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            _lib.reset_launch_count()
            loss = run()
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - base
            launches = _lib.launch_count()
            ms = _timed(run, args.reps, flush)
            nbytes = (FWD_BYTES + BWD_BYTES) * N * H * W
            res[arm] = {"ms_fwd_bwd": ms, "peak_extra_bytes": int(peak), "achieved_GBps": nbytes / (ms * 1e-3) / 1e9,
                        "loss": float(loss.detach()), "megreader_b200_launches": launches}
        emit({"bench": "db_loss", "N": N, "H": H, "W": W, "reps": args.reps,
              "timing": "CUDA events around each forward+backward, L2 flushed (256 MB write) before every call",
              "algorithmic_bytes": {"forward_per_sample_pixel": FWD_BYTES, "backward_per_sample_pixel": BWD_BYTES,
                                    "total": (FWD_BYTES + BWD_BYTES) * N * H * W},
              "kernels": res["kernels"], "library": res["library"],
              "speedup": res["library"]["ms_fwd_bwd"] / res["kernels"]["ms_fwd_bwd"],
              "loss_rel_diff": abs(res["kernels"]["loss"] - res["library"]["loss"]) / abs(res["library"]["loss"]),
              "one_NNHW_fp32_temporary_bytes": 4 * N * N * H * W, **gpu_info()})


def build_model(device, engine):
    """deformable_resnet50 + SegDetector(yaml args) as structure/model.py's BasicModel, name-seeded weights; engine=True puts every
    eligible convolution / transposed convolution / BatchNorm on megreader_b200.conv_engine (bf16 tcgen05 kernels)."""
    import megreader_b200
    megreader_b200.install_reference_api()
    import backbones
    import decoders
    from tests.weights import fill_state_dict

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.backbone = fill_state_dict(backbones.deformable_resnet50(pretrained=False), "dbb.")
            self.decoder = fill_state_dict(decoders.SegDetector(**YAML_HEAD), "dbd.")

        def forward(self, image):
            return self.decoder(self.backbone(image))

        def forward_library(self, image):
            return self.decoder._forward_framework(self.decoder._fuse(self.backbone(image)))
    net = Net().to(device).train()
    if engine:
        from megreader_b200 import conv_engine
        conv_engine.use_engine_convs(net)
    return net


def make_step(net, engine, batch_static, lr=0.007):
    """One training step (zero grads, forward, loss, backward, SGD) on `batch_static`; returns (step_fn, loss tensor getter)."""
    import decoders
    from oracle import db_port
    crit = decoders.L1BalanceCELoss()
    opt = torch.optim.SGD(net.parameters(), lr=lr, momentum=0.9, weight_decay=1e-4)

    def fwd_bwd():
        opt.zero_grad(set_to_none=True)
        if engine:
            loss, _ = crit(net(batch_static["image"]), batch_static)
        else:
            loss, _ = db_port.l1_balance_ce_loss(net.forward_library(batch_static["image"]), batch_static)
        loss.backward()
        return loss

    def step():
        loss = fwd_bwd()
        opt.step()
        return loss
    return step, fwd_bwd, opt


def bench_step(args, emit):
    dev = torch.device("cuda:0")
    H = W = 640
    for N in (2, 16):
        batch = synth_batch(7 + N, N, H, W, dev)
        out = {"bench": "db_step", "N": N, "H": H, "W": W, "steps": args.steps, "warmup": args.warmup}
        losses = {}
        for arm, engine in (("engine", True), ("library", False)):
            torch.manual_seed(0)
            net = build_model(dev, engine)
            static = {k: v.clone() for k, v in batch.items()}
            step, fwd_bwd, _ = make_step(net, engine, static)
            state = {k: v.clone() for k, v in net.state_dict().items()}
            # loss on the first batch from the initial weights (both arms): the comparison figure
            losses[arm] = float(fwd_bwd().detach())
            net.load_state_dict(state)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(max(3, args.warmup)):
                    step()
            torch.cuda.current_stream().wait_stream(side)
            graph, mode = None, "eager"
            if engine:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    static_loss = step()
                mode = "step captured in one CUDA graph"
            run = graph.replay if graph is not None else step
            for _ in range(2):
                run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                run()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            out[arm] = {"ms_per_step": ms, "images_per_s": N / (ms * 1e-3), "launch_mode": mode,
                        "peak_bytes": int(torch.cuda.max_memory_allocated())}
            if engine:
                out[arm]["finite_loss_after_steps"] = bool(torch.isfinite(static_loss).item())
            del net, graph
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
        out["loss_first_batch"] = losses
        out["loss_rel_delta_engine_vs_library"] = abs(losses["engine"] - losses["library"]) / abs(losses["library"])
        out["speedup"] = out["library"]["ms_per_step"] / out["engine"]["ms_per_step"]
        out["timing"] = "CUDA events around %d consecutive steps after warm-up" % args.steps
        out.update(gpu_info())
        emit(out)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("what", nargs="*", choices=["loss", "step"], default=[])
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_db.py needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    def emit(obj):
        print(json.dumps(obj), flush=True)
    what = args.what or ["loss", "step"]
    if "loss" in what:
        bench_loss(args, emit)
    if "step" in what:
        bench_step(args, emit)


if __name__ == "__main__":
    main()
