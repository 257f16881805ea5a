#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native MegReader recognition hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): CRNN backbone + 2x BiLSTM + 1D CTC, synthetic 32x256 lines (gray replicated to
3 channels, SURVEY.md D2), batch 512 PER GPU (weak scaling), bf16 compute, one full training step per "step":
forward + backward + Adam (+ NCCL gradient all-reduce when N > 1).  Metric: text-lines/sec, whole job.

Prints ONE JSON line (rank 0).  Extra objects on that line:
  e2e          same metric through the public module API with HOST (pinned) inputs: the step's H2D copies and the
               D2H read of the loss are inside the timed region
  roofline     the dominant hand-written kernel, algorithmic bytes / CUDA-event time vs MEASURED_PEAKS.json
  ctc2d        second half of BASELINE.json's metric: 2D-CTC fwd+bwd GB/s at the cfg-3 shape, saturating batch
  cpu_baseline the oracle port of the same step timed on this box's host cores (bounded sample)
--dump-outputs DIR writes what the last timed step returned (rank 0), its loss and log-probabilities, as DIR/<name>.npy in
float32.  That step starts from the seeded initial parameters, which are put back just before it: the steps before it train
with split-K atomic weight gradients whose summation order varies from run to run, and Adam would carry that into the
parameters.  Its inputs therefore depend on the arguments only, and two builds run with the same arguments can be compared
output for output.
--impl reference runs only the CPU arm (oracle port = restatement of the reference's own CPU path; the python
reference itself cannot travel to the GPU box) and prints the same line shape with "impl": "reference".
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "text-lines/sec CRNN+CTC train step (fwd+bwd+Adam), 32x256 lines, batch 512/GPU"
BATCH_PER_GPU = 512
IMG_W = 256
T_COLS = IMG_W // 4 + 1          # 65
L_MAX = 16                       # SURVEY.md §8d: label length U{1..16} at cfg 2


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ---------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], 0, set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- data
def synth_batch(seed, n):
    from tests.weights import crnn_batch
    x, labels, lengths = crnn_batch(seed, n, IMG_W, L_MAX, T_COLS)
    return torch.from_numpy(x), torch.from_numpy(labels), torch.from_numpy(lengths)


def headline_config(batch, world):
    """the `config` object of the headline line; the reference arm (--impl reference) reports the SAME object: it times a bounded
    sample of this workload on the host cores and says so in cpu_baseline.sample"""
    return {"workload": "CRNN + 2xBiLSTM + 1D CTC train step (crnn.yaml model), 3x32x256 fp32 input, "
                        "bf16 autocast compute, Adam lr 1e-3", "batch_per_gpu": batch,
            "global_batch": batch * world, "T": T_COLS, "classes": 38, "parallelism": "dp%d" % world,
            "l2": "3 rotating input batches (50 MB each) + 33 MB params/grads/Adam state per step exceed reuse; "
                  "activations (>1 GB/step) far exceed the 126 MB L2"}


# ---------------------------------------------------------------------------------------------- our arm
def build_model(device):
    import megreader_b200
    megreader_b200.install_reference_api()
    import backbones
    import decoders
    from tests.weights import fill_state_dict

    class Net(torch.nn.Module):          # structure/model.py:16-24 BasicModel: decoder(backbone(x), **kw)
        def __init__(self):
            super().__init__()
            self.backbone = fill_state_dict(backbones.crnn_backbone(), "bb.")
            self.decoder = fill_state_dict(decoders.CRNNDecoder(in_channels=512, inner_channels=256), "dec.")

        def forward(self, images, targets, lengths):
            return self.decoder(self.backbone(images), targets=targets, lengths=lengths, train=True)
    return Net().to(device).train()


def run_ours(args):
    import torch.distributed as dist
    import megreader_b200
    from megreader_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cudnn.benchmark = True                      # train.py:68
    torch.manual_seed(0)
    net = build_model(dev)
    model = net
    params = list(net.parameters())
    initial = [p.detach().clone() for p in params] if args.dump_outputs else None
    opt = torch.optim.Adam(params, lr=1e-3, fused=True, capturable=True)   # optimizer_scheduler.py:17-22, lr crnn.yaml
    from megreader_b200 import crnn_engine, dp
    crnn_engine.set_compute_dtype(torch.bfloat16)          # BASELINE.json cfg 2: bf16 compute, fp32 master weights
    batch = BATCH_PER_GPU // world if args.strong else BATCH_PER_GPU      # --strong: the reference's split (data_loader.py:40-43)
    # N > 1: the gradients are views into one flat buffer (decoder first = backward order): autograd accumulates into it, ONE
    # in-place NCCL all-reduce (AVG) runs between the two graphs, Adam reads the same views -- no flatten / divide / copy-back
    fg = dp.FlatGrads(list(net.decoder.parameters()) + list(net.backbone.parameters())) if world > 1 else None

    n_host = 3
    host = []
    for i in range(n_host):
        x, y, l = synth_batch(100 * rank + i, batch)
        host.append((x.pin_memory(), y.pin_memory(), l.pin_memory()))
    dev_batches = [tuple(t.to(dev) for t in hb) for hb in host]
    static = tuple(torch.empty_like(t) for t in dev_batches[0])

    def fwd_bwd(x, y, l):
        if fg is not None:
            fg.zero()                                      # one memset; the .grad views stay attached
        else:
            opt.zero_grad(set_to_none=True)
        loss, pred = model(x, y, l)
        loss.mean().backward()
        return loss, pred

    def eager_step(x, y, l):
        loss, _ = fwd_bwd(x, y, l)
        if fg is not None:
            fg.allreduce_()                                # NCCL all-reduce(AVG), in place on the flat 33 MB buffer
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def note(msg):
        if os.environ.get("MR_BENCH_VERBOSE"):
            print("[rank %d] %s" % (rank, msg), file=sys.stderr, flush=True)

    # warm up eagerly (cuBLAS workspaces, allocator, NCCL communicator), then capture the training step in CUDA
    # graphs: ~700 small launches per step would otherwise be bound by host launch overhead.  With N > 1 the
    # gradient all-reduce stays OUTSIDE the graphs (graph A = forward + backward, NCCL all-reduce, graph B = Adam).
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(3):
            eager_step(*dev_batches[i % n_host])
    torch.cuda.current_stream().wait_stream(side)
    barrier()
    note("eager warm-up done")
    _lib.reset_launch_count()
    graph_a = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph_a):
        static_loss, static_pred = fwd_bwd(*static)
        if world == 1:
            opt.step()
    graph_b = None
    if world > 1:
        graph_b = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph_b, pool=graph_a.pool()):
            opt.step()
    launches_per_step = _lib.launch_count()
    note("graphs captured")

    def step(x, y, l):
        for dst, src in zip(static, (x, y, l)):
            dst.copy_(src, non_blocking=True)
        graph_a.replay()
        if graph_b is not None:
            fg.allreduce_()
            graph_b.replay()
        return static_loss

    # ---- device-resident arm ("value")
    for i in range(args.warmup):
        step(*dev_batches[i % n_host])
    barrier()
    note("graph warm-up done")
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reset = None                                           # events around the parameter reset: its time is not step time
    e0.record()
    for i in range(args.steps):
        if initial is not None and i == args.steps - 1:
            reset = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reset[0].record()
            with torch.no_grad():
                for p, p0 in zip(params, initial):
                    p.copy_(p0)
            reset[1].record()
        loss = step(*dev_batches[i % n_host])
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": static_loss, "log_probs": static_pred})
    launches = launches_per_step * args.steps          # kernels of this library inside the replayed graphs
    ms = e0.elapsed_time(e1) - (reset[0].elapsed_time(reset[1]) if reset else 0.0)
    clocks = sampler.stop() if sampler else None
    final_loss = float(loss.mean().item())

    # ---- end-to-end arm: host pinned inputs, prefetch on a copy stream, loss read back every step
    copy_stream = torch.cuda.Stream()
    h2d = sum(t.numel() * t.element_size() for t in host[0])

    def fetch(i):
        with torch.cuda.stream(copy_stream):
            b = tuple(t.to(dev, non_blocking=True) for t in host[i % n_host])
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return b, ev

    def e2e_loop(k):
        nxt = fetch(0)
        last = None
        for i in range(k):
            (x, y, l), ev = nxt
            torch.cuda.current_stream().wait_event(ev)
            if i + 1 < k:
                nxt = fetch(i + 1)
            loss = step(x, y, l)
            last = float(loss.mean().item())        # D2H read of the step's result (4 bytes) each step
        return last
    e2e_loop(max(3, args.warmup))
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    e2e_loop(args.steps)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    lines = batch * world * args.steps
    if fg is not None and not fg.attached():
        raise SystemExit("gradient views were detached from the flat all-reduce buffer: the timed steps reduced stale data")
    out = {
        "metric": METRIC, "value": lines / (ms / 1e3), "unit": "lines/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.strong else "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": headline_config(batch, world),
        "e2e": {"value": lines / (ms_e2e / 1e3), "unit": "lines/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "final_loss": final_loss, "clocks": clocks,
    }
    if args.dump_outputs:
        out["dump_outputs"] = {"dir": args.dump_outputs, "files": ["loss.npy", "log_probs.npy"],
                               "last_step": "started from the seeded initial parameters (the reset before it is excluded from "
                                            "ms_per_step); final_loss is that step's loss"}
    if crnn_engine.LAST_LSTM_FLAGS is not None:            # error word of the persistent LSTM kernels (0 = no wait timed out)
        out["lstm_seq_err"] = int(crnn_engine.LAST_LSTM_FLAGS[-1])
        if out["lstm_seq_err"]:
            raise SystemExit("persistent LSTM kernel reported an inter-CTA wait time-out: results invalid")
    if rank == 0:
        out["ctc2d"], ctc_roof = bench_ctc2d(dev)
        out["roofline"] = bench_conv_roofline(dev)
        out["roofline_ctc2d"] = ctc_roof
        try:
            out["roofline_dcn"] = bench_dcn(dev)
        except Exception as e:                                # an extra arm never takes the headline down, but says why
            out["roofline_dcn"] = {"error": str(e)[:200]}
        try:
            out["input_step"] = bench_input_step(dev)
        except Exception as e:
            out["input_step"] = {"error": str(e)[:200]}
        try:
            out["parity"] = bench_parity(dev, lambda: net)
        except Exception as e:
            out["parity"] = {"error": str(e)[:200]}
        if os.environ.get("MR_BENCH_SKIP_CPU"):                 # profiling runs (ncu launch lists) skip the host-core arms
            out["cpu_baseline"] = {"skipped": "MR_BENCH_SKIP_CPU"}
        else:
            out["cpu_baseline"] = cpu_arm(steps=3, warmup=1, sample_n=16)
            try:
                out["cpu_baselines_other"] = cpu_side_baselines()
            except Exception as e:
                out["cpu_baselines_other"] = {"error": str(e)[:200]}
        out["stages"] = {"conv": "megreader_b200 tcgen05 implicit-GEMM kernels (fprop, dgrad, wgrad); conv0 (Cin=3): im2col kernel + cuBLAS",
                         "bias+ReLU+MaxPool, BatchNorm": "megreader_b200 CUDA (fused NHWC kernels)",
                         "BiLSTM+Linear": "recurrence: megreader_b200 persistent tcgen05 kernels (one launch per layer and pass, mode '%s'); "
                                          "input projections / Linear / weight-gradient GEMMs: cuBLAS" % crnn_engine.LSTM_MODE,
                         "conv weight gradients": "side stream, overlapped with the backward chain" if crnn_engine.WGRAD_SIDE_STREAM else "main stream",
                         "log_softmax+CTC": "megreader_b200 CUDA", "Adam": "library (torch fused, capturable)",
                         "allreduce": "one in-place NCCL all-reduce (AVG) of the flat gradient buffer the .grad views live in; no "
                                      "flatten / divide / copy-back launches" if world > 1 else "n/a",
                         "launch": "step captured in CUDA graph(s); the NCCL all-reduce runs between two graphs when N > 1"}
        emit_json(out)
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT = 64 << 20


def dump_outputs(path, arrays):
    """arrays: name -> device tensor, written as path/<name>.npy in float32 (at most DUMP_LIMIT bytes in all)"""
    total = sum(t.numel() * 4 for t in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------- 2D-CTC micro arm
def _graph_time(fn, iters=20):
    """device time of one call without the host launch gap: `iters` calls captured in a CUDA graph, replayed once"""
    fn(); fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3 / iters


def bench_ctc2d(dev, iters=10):
    """cfg-3 shape (T32,H8,C38,S32) fwd+bwd through ops.ctc_loss_2d's training pair at N in {32, 256, 2048, 16384}
    (SURVEY.md section 8d).  N = 16384: inputs (637 MB) exceed L2, CUDA events around back-to-back launches.  Smaller batches fit
    in L2 and a single launch is shorter than the host's launch gap, so they are timed as 20 launches inside one CUDA graph.
    Algorithmic bytes: SURVEY.md section 8(d) '3*|lp| + 2*iota + 12' = 117,292 B/sample."""
    from megreader_b200 import ctc2d
    from tests.cases import ctc2d_case
    T, H, C, S = 32, 8, 38, 32
    lp_b, idx_b = T * H * C * 4, 8 * S + 16
    fwd_bytes, bwd_bytes, pair_bytes = lp_b + T * C * 4 + idx_b + 4, 2 * lp_b + T * C * 4 + 4, 3 * lp_b + 2 * idx_b + 12
    pk = peaks()
    base = 256
    lp0, tg0, il0, tl0 = ctc2d_case(3, T, H, base, C, S, 12)
    sweep = {}
    ctc = roof = None
    for N in (32, 256, 2048, 16384):
        rep = max(1, N // base)
        sl = slice(0, min(N, base))
        d_lp = torch.from_numpy(np.ascontiguousarray(np.tile(lp0[:, :, sl], (1, 1, rep, 1)))).to(dev)
        d_tg = torch.from_numpy(np.tile(tg0[sl], (rep, 1))).to(dev)
        d_il = torch.from_numpy(np.tile(il0[sl], rep)).to(dev)
        d_tl = torch.from_numpy(np.tile(tl0[sl], rep)).to(dev)
        go = 1.0 / d_tl.float()
        fwd = lambda: ctc2d.ctc2d_forward_train(d_lp, d_tg, d_il, d_tl, 0)  # noqa: E731
        _, gf = fwd()
        bwd = lambda: ctc2d.ctc2d_backward_apply(go, d_lp, gf)  # noqa: E731
        if N < 16384:
            tf, tb = _graph_time(fwd), _graph_time(bwd)
            how = "20 launches in one CUDA graph (inputs L2-resident)"
        else:
            for _ in range(3):
                fwd(); bwd()
            torch.cuda.synchronize()
            tf = tb = 0.0
            for _ in range(iters):
                a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                a.record(); fwd(); b.record(); bwd(); c.record()
                torch.cuda.synchronize()
                tf += a.elapsed_time(b); tb += b.elapsed_time(c)
            tf, tb = tf / iters * 1e-3, tb / iters * 1e-3
            how = "CUDA events, back-to-back launches, inputs exceed L2"
        sweep[str(N)] = {"fwd_us": tf * 1e6, "bwd_us": tb * 1e6, "fwd_bwd_GBps": N * pair_bytes / (tf + tb) / 1e9,
                         "frac_of_hbm_peak": N * pair_bytes / (tf + tb) / 1e9 / pk["hbm_gbs"], "timing": how}
        if N == 16384:
            ctc = {"shape": {"T": T, "H": H, "C": C, "S": S, "N": N}, "fwd_us": tf * 1e6, "bwd_us": tb * 1e6,
                   "alg_bytes_per_sample_fwd_bwd": pair_bytes, "fwd_bwd_GBps": N * pair_bytes / (tf + tb) / 1e9,
                   "frac_of_hbm_peak": N * pair_bytes / (tf + tb) / 1e9 / pk["hbm_gbs"], "peak_source": pk["source"]}
            roof = {"kernel": "ctc2d_dp4_kernel<FAC> (2D-CTC training forward: Q, interleaved alpha/beta sweeps, factors)",
                    "bound": "hbm", "achieved": N * fwd_bytes / tf / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": N * fwd_bytes / tf / 1e9 / pk["hbm_gbs"], "traffic": _measured("ctc2d_dp4", "dram_bytes_per_launch"),
                    "peak_source": pk["source"], "alg_bytes_per_launch": N * fwd_bytes,
                    "note": "2D-CTC training forward (BASELINE.json metric, second half)"}
            # head epilogue in front of the loss (decoders/ctc_decoder2d.py:37-45): logits -> log_probs, and the fused backward
            try:
                from megreader_b200 import ctc2d_head
                m = torch.randn(N, 1, H, T, device=dev)
                z = torch.randn(N, C, H, T, device=dev)
                for _ in range(2):
                    ctc2d_head.head_forward(m, z); ctc2d_head.head_backward(m, z, gfac=gf, grad_out=go)
                a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                a.record()
                for _ in range(iters):
                    ctc2d_head.head_forward(m, z)
                b.record()
                for _ in range(iters):
                    ctc2d_head.head_backward(m, z, gfac=gf, grad_out=go)
                c.record()
                torch.cuda.synchronize()
                hf, hb = a.elapsed_time(b) / iters * 1e-3, b.elapsed_time(c) / iters * 1e-3
                ctc["head_epilogue"] = {"fwd_us": hf * 1e6, "bwd_factored_us": hb * 1e6,
                                        "fwd_GBps": N * (2 * lp_b + H * T * 4) / hf / 1e9,
                                        "bwd_GBps": N * (2 * lp_b + T * C * 4) / hb / 1e9,
                                        "fwd_frac_of_hbm_peak": N * (2 * lp_b + H * T * 4) / hf / 1e9 / pk["hbm_gbs"],
                                        "bwd_frac_of_hbm_peak": N * (2 * lp_b + T * C * 4) / hb / 1e9 / pk["hbm_gbs"]}
                del m, z
            except Exception as e:
                ctc["head_epilogue"] = {"error": str(e)[:200]}
        del d_lp, gf
    ctc["batches"] = sweep
    return ctc, roof


def _measured(kernel, key):
    """A number taken from the committed ncu summary of the current revision (profiles/measured_r2.json, written from the
    `ncu --set full` captures listed in profiles/); None when no capture of that kernel is committed."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "measured_r2.json")))
        return d[kernel][key]
    except Exception:
        return None


def bench_dcn(dev, iters=10):
    """DCNv2 forward at SURVEY.md section 8d's shapes (B = 8): fused tcgen05 implicit GEMM (csrc/dcn_tcgen05.cu), timed through the
    autograd surface (NHWC copy + weight pack + the GEMM).  Roofline: tensor pipe, 2*C*9*Cout*Ho*Wo flops per sample."""
    from megreader_b200 import dcn
    pk = peaks()
    out = {}
    for C, H in ((128, 64), (256, 32), (512, 16)):
        B = 8
        x = torch.randn(B, C, H, H, device=dev)
        w = torch.randn(C, C, 3, 3, device=dev) / (3 * C ** 0.5)
        off = 2 * torch.randn(B, 18, H, H, device=dev)
        m = torch.sigmoid(torch.randn(B, 9, H, H, device=dev))
        fn = lambda: dcn.modulated_deform_conv(x, off, m, w, None, 1, 1, 1, 1, 1)  # noqa: E731
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        sec = a.elapsed_time(b) / iters * 1e-3
        # backward through the reference's pybind-style entry (deform_conv_cuda.cpp:566-679): fused weight + data gradient kernels
        go = torch.randn(B, C, H, H, device=dev)
        gi, gw, goff, gm = torch.zeros_like(x), torch.zeros_like(w), torch.zeros_like(off), torch.zeros_like(m)
        bw = lambda: dcn.modulated_deform_conv_cuda_backward(x, w, None, None, off, m, None, gi, gw, None, goff, gm, go,  # noqa: E731
                                                            3, 3, 1, 1, 1, 1, 1, 1, 1, 1, False)
        for _ in range(3):
            bw()
        torch.cuda.synchronize()
        a.record()
        for _ in range(iters):
            bw()
        b.record()
        torch.cuda.synchronize()
        bsec = a.elapsed_time(b) / iters * 1e-3
        flops = 2.0 * B * C * 9 * C * H * H
        out["C%d@%dx%d" % (C, H, H)] = {"fwd_us": sec * 1e6, "alg_TFLOPs": flops / sec / 1e12,
                                        "frac_of_tensor_peak": flops / sec / 1e12 / pk["bf16_tflops"],
                                        "mma_TFLOPs_issued": 3 * flops / sec / 1e12,
                                        "bwd_us": bsec * 1e6, "bwd_alg_TFLOPs": 2 * flops / bsec / 1e12,
                                        "bwd_frac_of_tensor_peak": 2 * flops / bsec / 1e12 / pk["bf16_tflops"]}
    return {"kernel": "dcn_fwd_tcgen05_kernel (bilinear gather = A-operand producer, bf16 hi/lo split: 3 MMAs per K block); backward = "
                      "dcn_wgrad_tcgen05_kernel + dcn_dgrad_tcgen05_kernel (no column matrices in HBM)",
            "bound": "tensor", "unit": "TFLOP/s", "peak": pk["bf16_tflops"], "peak_source": pk["source"], "B": 8, "shapes": out,
            "traffic_bwd_C128@64x64": {"dcn_dgrad_tcgen05_kernel": _measured("dcn_dgrad_c128", "dram_bytes_per_launch"),
                                       "dcn_wgrad_tcgen05_kernel": _measured("dcn_wgrad_c128", "dram_bytes_per_launch")},
            "round1_fwd_us": {"C128@64x64": 319.2, "C256@32x32": 264.5, "C512@16x16": 215.3},
            "round1_fwd_bwd_us": {"C128@64x64": 1611.0, "C256@32x32": 1115.3, "C512@16x16": 944.9}}


def bench_input_step(dev, n=512, reps=5):
    """Input step of SURVEY.md section 8 row N3 on the GPU: a ragged batch of decoded uint8 HWC line images -> resize to 32x256,
    normalise, CHW fp32 (one launch) + label strings -> class indices (one launch).  `e2e` includes the host-side concatenation of
    the ragged batch and the pinned H2D copies; `device` is the two kernels alone (CUDA events)."""
    from megreader_b200 import input_pipeline as ip
    rng = np.random.RandomState(0)
    images = [rng.randint(0, 256, size=(int(rng.randint(24, 49)), int(rng.randint(60, 301)), 3), dtype=np.uint8) for _ in range(n)]
    alphabet = "0123456789abcdefghijklmnopqrstuvwxyz"
    texts = ["".join(alphabet[int(c)] for c in rng.randint(0, 36, size=int(rng.randint(1, 17)))) for _ in range(n)]
    for _ in range(2):
        ip.resize_normalize(images, (32, IMG_W), "resize", dev); ip.pack_labels(texts, None, 32, dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        x = ip.resize_normalize(images, (32, IMG_W), "resize", dev)
        y, l = ip.pack_labels(texts, None, 32, dev)
    torch.cuda.synchronize()
    e2e = (time.perf_counter() - t0) / reps
    src_bytes = sum(im.size for im in images)
    return {"batch": n, "e2e_lines_per_s": n / e2e, "e2e_ms": e2e * 1e3, "src_bytes": src_bytes, "out_bytes": int(x.numel() * 4),
            "note": "host: numpy concatenation of the ragged uint8 batch + pinned copies; device: csrc/input_pipeline.cu; JPEG "
                    "decode and the LMDB read stay on the host (not timed)"}


def bench_parity(dev, model_fn):
    """bf16 engine (the timed mode) against the fp32 engine on one 512-line bench batch: what tests/test_bench_shape_parity_gpu.py
    asserts, recomputed live."""
    from megreader_b200 import crnn_engine
    net = model_fn()
    x, y, l = [t.to(dev) for t in synth_batch(0, BATCH_PER_GPU)]
    state = {k: v.clone() for k, v in net.state_dict().items()}
    res = {}
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        crnn_engine.set_compute_dtype(dt)
        with torch.no_grad():
            net.train()
            loss, lp = net(x, y, l)
        net.load_state_dict(state)
        res[name] = (float(loss), lp.float())
    crnn_engine.set_compute_dtype(torch.bfloat16)
    l32, p32 = res["fp32"]
    l16, p16 = res["bf16"]
    dmax = float((p16 - p32).abs().max())
    top2 = p32.topk(2, dim=2).values
    decided = (top2[..., 0] - top2[..., 1]) > 4 * dmax
    same = p16.argmax(2) == p32.argmax(2)
    return {"shape": "N=512, 3x32x256, T=65", "loss_rel_delta_bf16_vs_fp32": abs(l16 - l32) / abs(l32),
            "max_abs_logprob_delta": dmax, "argmax_agreement": float(same.float().mean()),
            "argmax_agreement_where_fp32_margin_gt_4x_delta": float(same[decided].float().mean()) if bool(decided.any()) else None,
            "decided_fraction": float(decided.float().mean()),
            "fp32_engine_vs_cpu_oracle": "tests/test_bench_shape_parity_gpu.py (loss / log-probs 1e-4, labels bit-exact)"}


def bench_conv_roofline(dev, iters=10):
    """Dominant kernel of the step: conv_fprop_tcgen05_kernel (implicit-GEMM conv, also used for dgrad) at its largest
    shape (conv5: 512 x 4 x 65 x 512 -> 512 ch, 3x3), timed alone with CUDA events; inputs 136 MB + output 136 MB
    exceed L2.  Algorithmic FLOPs = 2 * P * Cout * kh*kw*C per launch; peak = measured cuBLAS bf16 burst."""
    from megreader_b200 import nnops
    N, H, W, C, Cout, k, p = BATCH_PER_GPU, 4, 65, 512, 512, 3, 1
    x = torch.randn(N, H, W, C, device=dev).bfloat16()
    wm = (torch.randn(Cout, k * k * C, device=dev) / 68).bfloat16()
    for _ in range(3):
        nnops.conv_fprop_tc(x, wm, k, k, p, p)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        nnops.conv_fprop_tc(x, wm, k, k, p, p)
    b.record()
    torch.cuda.synchronize()
    sec = a.elapsed_time(b) / iters * 1e-3
    flops = 2.0 * N * H * W * Cout * k * k * C
    pk = peaks()
    return {"kernel": "conv_fprop_tcgen05_kernel<256,2,1,1> (implicit-GEMM 3x3 conv via 4-D TMA, conv5 shape, bf16 in / fp32 acc)",
            "bound": "tensor", "achieved": flops / sec / 1e12, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
            "frac": flops / sec / 1e12 / pk["bf16_tflops"],
            "traffic": _measured("conv_fprop_conv5", "dram_bytes_per_launch"),   # ncu --set full of this revision, or None
            "traffic_algorithmic": 2.0 * N * H * W * C + 2.0 * N * H * W * Cout + 2.0 * Cout * k * k * C,
            "peak_source": pk["source"],
            "alg_flops_per_launch": flops, "us_per_launch": sec * 1e6}


# ---------------------------------------------------------------------------------------------- CPU / reference arm
def usable_cores():
    """Host threads this process can really use: affinity mask and cgroup CPU quota (os.cpu_count() reports the
    whole machine inside a quota-limited container and oversubscribing it is 100x slower), capped at 32 because
    the ATen CPU kernels of this small model stop scaling there."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        pass
    return max(1, min(n, 32))


def cpu_arm(steps, warmup, sample_n, budget_s=25.0):
    """The reference's own CPU path for this workload, restated by oracle/crnn_port.py (validated bit-for-bit against
    the unmodified reference modules in the build container): fp32, all host cores, same model/optimizer.  With a budget
    (seconds) the warm-up stops after half of it and the timed steps after all of it; budget_s=None runs every step."""
    from oracle import crnn_port
    from tests.weights import fill_state_dict
    cores = usable_cores()
    torch.set_num_threads(cores)
    bb = fill_state_dict(crnn_port.CRNNBackbonePort(), "bb.").train()
    dec = fill_state_dict(crnn_port.CRNNDecoderPort(), "dec.").train()
    opt = torch.optim.Adam(list(bb.parameters()) + list(dec.parameters()), lr=1e-3)
    x, y, l = synth_batch(0, sample_n)

    def step():
        opt.zero_grad()
        loss, _ = dec(bb(x), y, l, train=True)
        loss.mean().backward()
        opt.step()
        return loss
    tw = time.perf_counter()
    for _ in range(warmup):
        step()
        if budget_s is not None and time.perf_counter() - tw > budget_s / 2:
            break
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        step()
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    steps = done
    dt = time.perf_counter() - t0
    return {"value": sample_n * steps / dt, "unit": "lines/s", "cores": cores, "kind": "port",
            "sample": "%d steps of a %d-line batch (3x32x256 fp32) of the same train step, torch CPU fp32, %d threads"
                      % (steps, sample_n, torch.get_num_threads()), "ms_per_step": dt / steps * 1e3}


def cpu_side_baselines():
    """BASELINE.md section 3's remaining CPU figures, on this box's host cores (single thread for the C restatements):
    cfg 1 exactly (CRNN + BiLSTM + 1D CTC, N = 4, 3x32x100, fwd + bwd + Adam) through the oracle port; the fp64 C restatement of the
    2D-CTC kernels (K1 + K2 + K3) at the cfg-3 shape, N in {32, 256}; the fp64 C restatement of DCNv2 forward / backward at the three
    bench shapes for ONE sample (the GPU figures in roofline_dcn are for B = 8)."""
    import statistics
    from oracle import capi, crnn_port
    from tests.cases import ctc2d_case
    from tests.weights import crnn_batch, fill_state_dict
    out = {"cores_c_restatements": 1}
    # cfg 1
    cores = usable_cores()
    torch.set_num_threads(cores)
    bb = fill_state_dict(crnn_port.CRNNBackbonePort(), "bb.").train()
    dec = fill_state_dict(crnn_port.CRNNDecoderPort(), "dec.").train()
    opt = torch.optim.Adam(list(bb.parameters()) + list(dec.parameters()), lr=1e-3)
    x, y, l = (torch.from_numpy(a) for a in crnn_batch(0, 4, 100, 8, 26))
    ts = []
    for i in range(7):
        t0 = time.perf_counter()
        opt.zero_grad()
        loss, _ = dec(bb(x), y, l, train=True)
        loss.mean().backward()
        opt.step()
        if i >= 2:
            ts.append(time.perf_counter() - t0)
    out["cfg1_crnn_ctc_n4_32x100"] = {"lines_per_s_median": 4 / statistics.median(ts), "lines_per_s_best": 4 / min(ts), "threads": cores,
                                       "kind": "port", "timed_steps": len(ts)}
    # 2D-CTC, fp64 restatement of the reference kernels
    c2 = {}
    for N in (32, 256):
        lp, tg, il, tl = ctc2d_case(3, 32, 8, N, 38, 32, 12)
        go, lp64 = (1.0 / tl).astype(np.float64), lp.astype(np.float64)
        ts = []
        for i in range(3 if N == 32 else 2):
            t0 = time.perf_counter()
            capi.ctc2d_fwd_bwd(go, lp64, tg, il, tl)
            ts.append(time.perf_counter() - t0)
        c2[str(N)] = {"fwd_bwd_ms_best": min(ts) * 1e3, "samples_per_s": N / min(ts)}
    out["ctc2d_oracle_f64_T32_H8_C38_S32"] = c2
    # DCNv2, fp64 restatement, one sample
    rng = np.random.RandomState(0)
    dc = {}
    for C, H in ((128, 64), (256, 32), (512, 16)):
        x = rng.standard_normal((1, C, H, H))
        w = rng.standard_normal((C, C, 3, 3)) / (3 * C ** 0.5)
        off = 2 * rng.standard_normal((1, 18, H, H))
        m = 1 / (1 + np.exp(-rng.standard_normal((1, 9, H, H))))
        t0 = time.perf_counter()
        o = capi.dcn_forward(x, w, None, off, m)
        t1 = time.perf_counter()
        capi.dcn_backward(x, w, None, off, m, rng.standard_normal(o.shape))
        t2 = time.perf_counter()
        dc["C%d@%dx%d" % (C, H, H)] = {"fwd_ms_per_sample": (t1 - t0) * 1e3, "bwd_ms_per_sample": (t2 - t1) * 1e3}
    out["dcn_oracle_f64_one_sample"] = dc
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = 32
    res = cpu_arm(steps=args.steps, warmup=args.warmup, sample_n=n, budget_s=None)     # --steps is the number of timed steps
    out = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": "lines/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": headline_config(BATCH_PER_GPU, max(1, args.gpus)),
           "sample": "each step = a %d-line bounded sample of the 512-line batch, fp32 on the host cores (the reference's CPU path "
                     "has no bf16 autocast)" % n,
           "cpu_baseline": res,
           "e2e": {"value": res["value"], "unit": "lines/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_json(out)


class _QuietStdout:
    """The contract is ONE JSON line on stdout: libraries that write to file descriptor 1 on their own (NCCL prints its
    version banner there at communicator init) are sent to stderr; `emit` writes the line to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self._real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.write(self._real, (line + "\n").encode())


_OUT = None


def emit_json(obj):
    line = json.dumps(obj)
    if _OUT is not None:
        _OUT.emit(line)
    else:
        print(line, flush=True)


def main():
    global _OUT
    _OUT = _QuietStdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json configuration: 2 = CRNN + 1D CTC (headline, default); 3 = ResNet50-PPM + 2D CTC; "
                         "4 = FPN50 + attention decoder; 5 = deformable ResNet50 + FPN + EAST (bench_trunks.py)")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch for --config 3 / 4 (default 32)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's loss and log-probabilities as DIR/<name>.npy; that "
                         "step starts from the seeded initial parameters (headline workload only)")
    ap.add_argument("--strong", action="store_true",
                    help="reference semantics (data/data_loader.py:40-43): global batch 512 split over the ranks (strong scaling) "
                         "instead of 512 per GPU")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != 2):
        ap.error("--dump-outputs is implemented for the headline workload (--impl ours --config 2)")
    if args.impl == "reference":
        run_reference(args)
    elif args.config != 2:
        import bench_trunks
        bench_trunks.run(args, peaks(), ClockSampler, emit_json)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
