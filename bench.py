#!/usr/bin/env python
"""Benchmark of the hot path: ViT-B/16 224 px, patches serialised along the generalised Hilbert curve (14 x 14 grid),
one TRAINING step = forward + soft-target CE + backward + (DP gradient all-reduce) + grad-norm clip + AdamW, bf16
parameters/activations (main.py:157), dropout active, synthetic images and random-init weights.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch B] [--config vit_b16_224]
                    [--dump-outputs DIR]

N > 1: launched by the driver as `python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...`.
Prints ONE JSON line on rank 0 (contract in the task statement): `value` = images/s over all GPUs with inputs resident
in HBM; `e2e` = same metric through the public API with pinned-host inputs copied H2D (and the loss read back) inside
the timed region; `roofline` for the dominant kernel family (tcgen05 GEMM), timed live with CUDA events;
`cpu_baseline` = the CPU oracle port of the reference path on this box's host cores (N = 1 only).
`--impl reference` times that CPU port alone (all host threads, a bounded batch per step).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PK = os.path.join(ROOT, "space-filling-curves-for-vision-transformers_b200")
for p in (ROOT, PK):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

CONFIGS = {
    # name: img, patch, D, depth, heads, mlp, classes, default per-GPU batch
    "vit_b16_224": dict(img=224, patch=16, D=768, depth=12, heads=12, mlp=3072, classes=1000, batch=256),
    "vit_s16_224": dict(img=224, patch=16, D=384, depth=12, heads=6, mlp=1536, classes=1000, batch=256),
    "vit_l16_384": dict(img=384, patch=16, D=1024, depth=24, heads=16, mlp=4096, classes=1000, batch=64),
    "vit_tiny4_32": dict(img=32, patch=4, D=192, depth=12, heads=3, mlp=768, classes=10, batch=1024),
    # BASELINE.json configs[4]: 64 x 64 patch grid, 4096 tokens per image — inference only (--mode infer)
    "vit_b16_1024": dict(img=1024, patch=16, D=768, depth=12, heads=12, mlp=3072, classes=1000, batch=4),
}
METRIC = "ViT-B/16 224px Hilbert images/sec fwd+bwd"       # BASELINE.json's metric, quoted on vit_b16_224
CONFIG_LABEL = {"vit_b16_224": "ViT-B/16 224px", "vit_s16_224": "ViT-S/16 224px", "vit_l16_384": "ViT-L/16 384px",
                "vit_tiny4_32": "ViT-Tiny/4 32px", "vit_b16_1024": "ViT-B/16 1024px"}


def metric_name(config, curve, infer=False):
    """The metric string names the configuration it was measured on (only vit_b16_224 + hilbert is BASELINE.json's)."""
    if infer:
        return f"{CONFIG_LABEL[config]} {curve} images/sec fwd (bf16 inference)"
    return f"{CONFIG_LABEL[config]} {'Hilbert' if curve == 'hilbert' else curve} images/sec fwd+bwd"


def fwd_flops_per_image(c):
    """Algorithmic forward FLOPs (2mnk per GEMM, 4 N^2 D attention per layer) — SURVEY.md §8d / BASELINE.md §3."""
    N = (c["img"] // c["patch"]) ** 2
    D, M, K = c["D"], c["mlp"], 3 * c["patch"] ** 2
    pe = 2 * N * K * D
    layer = 2 * N * D * 3 * D + 4 * N * N * D + 2 * N * D * D + 2 * 2 * N * D * M
    head = 2 * N * D * 64 + 2 * (N * 64) * 2 * D + 2 * 2 * D * c["classes"]
    return pe + c["depth"] * layer + head


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_b200_model(c, device, curve="hilbert"):
    from src.curves import space_filling_curves as sc
    from src.models.vit import VisionTransformer
    from src.tokenizers.multiscale.multi_hilbert import SFCEmbedding1D
    from src.tokenizers.multiscale.multi_zigzag import RasterScan1DGroupedEmbedding
    torch.manual_seed(42)                                    # main.py:151-152
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)                  # main.py:157: parameters, buffers and optimizer state in bf16
    try:
        if curve == "raster":
            tok = RasterScan1DGroupedEmbedding(c["img"], c["patch"], 1, 3, c["D"])
        else:                                                             # embed-and-prune curve on the patch grid
            fn = {"hilbert": sc.hilbert_curve, "morton": sc.z_curve, "peano": sc.peano_curve, "moore": sc.moore_curve}[curve]
            tok = SFCEmbedding1D(c["img"], c["patch"], 1, 3, c["D"], curve_fn=fn)
        model = VisionTransformer(patch_embed=tok, depth=c["depth"], n_heads=c["heads"], mlp_dim=c["mlp"],
                                  num_classes=c["classes"]).to(device)
    finally:
        torch.set_default_dtype(prev)
    return model.train()


def build_oracle_model(c):
    from oracle import model as om
    torch.manual_seed(42)
    tok = om.SFCEmbedding1D(c["img"], c["patch"], 1, 3, c["D"], "hilbert")
    tok.n_patches = (c["img"] // c["patch"]) ** 2
    return om.VisionTransformer(tok, depth=c["depth"], n_heads=c["heads"], mlp_dim=c["mlp"], num_classes=c["classes"]).train()


def soft_targets(labels_a, labels_b, lam, classes):
    oh = torch.nn.functional.one_hot
    return lam * oh(labels_a, classes).float() + (1 - lam) * oh(labels_b, classes).float()


DUMP_SAMPLE = 1 << 22          # elements kept of a larger array (16 MB in float32): four arrays stay under 64 MB


def _host_sample(t):
    """`t` as float32 on the host. Beyond DUMP_SAMPLE elements: the flattened tensor at DUMP_SAMPLE sorted positions
    drawn from a fixed seed, so every run and every build of the same configuration keeps the same positions."""
    t = t.detach()
    if t.numel() > DUMP_SAMPLE:
        idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
        t = t.reshape(-1)[idx.to(t.device)]
    return t.float().cpu()


def step_outputs(logits, loss=None, model=None):
    """What a caller of the timed step holds after its last step, copied to the host: the logits, and for a training
    step the loss, the updated parameters and their gradients (each flattened and concatenated in model.parameters()
    order; a parameter without a gradient contributes zeros)."""
    out = {"logits": _host_sample(logits)}
    if loss is not None:
        out["loss"] = _host_sample(loss.reshape(1))
    if model is not None:
        params = list(model.parameters())
        out["params"] = _host_sample(torch.cat([p.detach().float().reshape(-1) for p in params]))
        out["grads"] = _host_sample(torch.cat([(torch.zeros_like(p) if p.grad is None else p.grad).float().reshape(-1)
                                               for p in params]))
    return out


def write_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def cpu_reference_throughput(c, steps, warmup, batch):
    """The reference path on the host CPU (oracle port: stock torch fp32 modules + C-oracle curve indices)."""
    torch.set_num_threads(os.cpu_count() or 1)
    model = build_oracle_model(c)
    opt = torch.optim.AdamW(model.parameters(), lr=3e-4, weight_decay=5e-5)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(batch, 3, c["img"], c["img"], generator=g)
    tgt = soft_targets(torch.randint(0, c["classes"], (batch,), generator=g), torch.randint(0, c["classes"], (batch,), generator=g), 0.3, c["classes"])
    from oracle.model import soft_target_cross_entropy
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        loss = soft_target_cross_entropy(model(x), tgt)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return batch / sec, sec, torch.get_num_threads()


def curve_generation_table(device):
    """K1 (csrc/curves.cu, one launch pair: count + emit) next to the CPU oracle port of the reference's
    embed_and_prune_sfc (C restatement of its float pipeline, 1 core) for the grids BASELINE.md §4 names. The reference's
    own Python recursion took 2.2 ms (n = 14) ... 9.0 s (n = 1024) at survey time (BASELINE.md §4, this container)."""
    from oracle import curves as oc
    from sfcvit import ops
    rows = []
    for curve, n in (("hilbert", 14), ("hilbert", 24), ("peano", 24), ("hilbert", 64), ("z", 224), ("hilbert", 224), ("hilbert", 1024)):
        ops.curve_perm(curve, n, n, device)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            perm, _inv = ops.curve_perm(curve, n, n, device)
        e1.record()
        torch.cuda.synchronize()
        gpu_us = e0.elapsed_time(e1) * 100.0                          # per call, microseconds
        t0 = time.perf_counter()
        ref = oc.flat_perm(curve, n, n)
        cpu_us = (time.perf_counter() - t0) * 1e6
        same = bool((perm.cpu().numpy().astype("int64") == ref).all())
        rows.append({"curve": curve, "n": n, "k1_us": round(gpu_us, 1), "cpu_oracle_us": round(cpu_us, 1), "bit_exact": same,
                     "cells_per_us_k1": round(n * n / gpu_us, 1)})
    return rows


def patch_embed_sweep(device, peaks):
    """BASELINE.json's second metric on the configurations where the bound really is HBM (SURVEY.md §8d): the fused
    curve-gather patch embed alone, fp32 NCHW input, embed-and-prune Hilbert order, CUDA events over rotating inputs
    (> L2 in total). Algorithmic bytes = image read once + token matrix written once."""
    from sfcvit import functional as SF
    from sfcvit import ops
    rows = []
    for name, img, p, D, B in (("vit_tiny4_32", 32, 4, 192, 1024), ("vit_tiny4_32 (B 8192)", 32, 4, 192, 8192),
                               ("vit_s16_224", 224, 16, 384, 256), ("vit_b16_224", 224, 16, 768, 256)):
        n = img // p
        perm, _ = ops.curve_perm("hilbert", n, n, device)
        g = torch.Generator(device=device).manual_seed(0)
        w = (torch.randn(D, 3 * p * p, generator=g, device=device) * 0.02).to(torch.bfloat16)
        wk = SF.kernel_weight(w, 3, p, 1, "p1p2c")
        bias = torch.zeros(D, dtype=torch.bfloat16, device=device)
        nbuf = max(2, min(16, int(400e6 // (B * 3 * img * img * 4)) + 1))
        xs = [torch.randn(B, 3, img, img, generator=g, device=device) for _ in range(nbuf)]
        out = torch.empty(B, n * n, D, dtype=torch.bfloat16, device=device)
        for i in range(3):
            ops.patch_embed_fwd(xs[i % nbuf], perm, wk, bias, p, 1, out=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 20
        e0.record()
        for i in range(iters):
            ops.patch_embed_fwd(xs[i % nbuf], perm, wk, bias, p, 1, out=out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        nbytes = B * 3 * img * img * 4 + B * n * n * D * 2
        flops = 2.0 * B * n * n * (3 * p * p) * D
        t_roof = max(nbytes / (peaks["hbm_gbs"] * 1e9), flops / (peaks["tf_sustained"] * 1e12)) * 1e3
        rows.append({"config": name, "batch": B, "ms": round(ms, 4), "achieved_gbs": round(nbytes / ms / 1e6, 1),
                     "frac_hbm": round(nbytes / ms / 1e6 / peaks["hbm_gbs"], 3), "frac_of_max_hbm_tensor_roofline": round(t_roof / ms, 3),
                     "bound": "hbm" if nbytes / (peaks["hbm_gbs"] * 1e9) > flops / (peaks["tf_sustained"] * 1e12) else "tensor"})
        del xs
    return rows


def torch_gpu_throughput(c, device, batch, steps, warmup, compiled=False, infer=False):
    """INFORMATIONAL comparator (SURVEY.md §8d): the reference's own modules (oracle port = stock torch nn.TransformerEncoder,
    SDPA, nn.Linear -> cuBLAS / cuDNN / flash kernels) on the SAME B200, bf16 autocast as the reference trains
    (train.py:155), eager or torch.compile(mode="reduce-overhead") as main.py:284. Same step as the b200 arm:
    forward + soft-target CE + backward + clip + AdamW. Library kernels: not the product, the kernel to beat."""
    from oracle.model import soft_target_cross_entropy
    model = build_oracle_model(c).to(device)
    fwd = torch.compile(model, mode="reduce-overhead") if compiled else model
    opt = torch.optim.AdamW(model.parameters(), lr=3e-4, weight_decay=5e-5, fused=True)
    g = torch.Generator(device=device).manual_seed(0)
    xs = [torch.randn(batch, 3, c["img"], c["img"], generator=g, device=device) for _ in range(4)]
    la = torch.randint(0, c["classes"], (batch,), generator=g, device=device)
    tgt = soft_targets(la, la.roll(1), 0.3, c["classes"])

    def step(x):
        if infer:
            with torch.no_grad(), torch.amp.autocast(device_type="cuda", dtype=torch.bfloat16):
                return fwd(x)
        opt.zero_grad(set_to_none=True)
        with torch.amp.autocast(device_type="cuda", dtype=torch.bfloat16):
            loss = soft_target_cross_entropy(fwd(x), tgt)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        return loss
    if infer:
        model.eval()
    for i in range(warmup):
        step(xs[i % 4])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(xs[i % 4])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    del model, opt, xs
    torch.cuda.empty_cache()
    return batch / (ms * 1e-3), ms


def run_torch_gpu_arm(args, c):
    """`--impl torch-gpu`: stock PyTorch on this GPU, eager and compiled, one JSON line (informational)."""
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl torch-gpu needs a CUDA device")
    if int(os.environ.get("RANK", "0")) != 0:
        return
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    B = args.batch or c["batch"]
    infer = args.mode == "infer"
    res = {}
    for name, comp in (("eager", False), ("compiled_reduce_overhead", True)):
        try:
            ips, ms = torch_gpu_throughput(c, device, B, args.steps, max(3, args.warmup), compiled=comp, infer=infer)
            res[name] = {"value": ips, "ms_per_step": ms}
        except Exception as e:                                        # e.g. no host compiler for inductor on the box
            res[name] = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
    best = max((v["value"] for v in res.values() if "value" in v), default=None)
    print(json.dumps({"metric": metric_name(args.config, args.curve, infer), "impl": "torch-gpu", "value": best, "unit": "images/s",
                      "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "dtype": "bf16 autocast (fp32 parameters)",
                      "data": "synthetic", "config": {"workload": f"{args.config} stock torch modules (oracle port of the reference) on the GPU", "batch_per_gpu": B},
                      "variants": res, "note": "library kernels (cuBLAS, flash SDPA, ATen); informational comparator, not the product"}), flush=True)


def run_reference_arm(args, c):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = args.cpu_batch
    infer = args.mode == "infer"
    if infer:
        ips, sec, threads, batch = cpu_reference_forward(c, args.steps, max(0, min(args.warmup, 1)), batch)
    else:
        ips, sec, threads = cpu_reference_throughput(c, args.steps, max(0, min(args.warmup, 1)), batch)
    line = {
        "metric": metric_name(args.config, args.curve, infer), "value": ips, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "impl": "reference",
        "config": {"workload": f"{args.config} Hilbert(embed-and-prune) " + ("inference forward" if infer else "train step fwd+bwd+clip+AdamW") + ", CPU oracle port of the reference path",
                   "batch_per_step": batch},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} steps of batch {batch} (fp32, {threads} threads)"},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_infer(args, c):
    """`--mode infer`: forward only (eval, no_grad, bf16 parameters), BASELINE.json configs[1] (ViT-S/16 224) and
    configs[4] (ViT-B/16 1024 px, 4096 tokens). Replicas only for N > 1 (no collective on the data path). The forward is
    replayed from one CUDA graph over rotating input batches; `roofline` is per kernel family (GEMM, attention, patch
    embed) from an eager replica timed with CUDA events around each launch."""
    import torch.distributed as dist
    from sfcvit import ops
    from src.training import distributed as D
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (B200); there is no CPU fallback")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    rank, world = D.init_from_env("nccl")
    B = args.batch or c["batch"]
    N = (c["img"] // c["patch"]) ** 2
    model = build_b200_model(c, device, args.curve).eval()
    g = torch.Generator(device=device).manual_seed(1234 + rank)
    img_bytes = B * 3 * c["img"] ** 2 * 4
    n_bufs = max(4, -(-3 * 126_000_000 // img_bytes))                  # rotating inputs: together > 3 x L2
    n_bufs = min(n_bufs, 64)
    dev_imgs = [torch.randn(B, 3, c["img"], c["img"], generator=g, device=device) for _ in range(n_bufs)]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    with torch.no_grad():
        for i in range(args.warmup):
            model(dev_imgs[i % n_bufs])
        sync_all()
        ops.GEMM_PROFILE, ops.PE_PROFILE, ops.ATTN_PROFILE = [], [], []
        roof_steps = min(3, max(1, args.steps))
        l0 = ops.LAUNCHES
        for i in range(roof_steps):
            model(dev_imgs[i % n_bufs])
        sync_all()
        launches_per_step = (ops.LAUNCHES - l0) // roof_steps
        gprof, ops.GEMM_PROFILE = ops.GEMM_PROFILE, None
        pprof, ops.PE_PROFILE = ops.PE_PROFILE, None
        aprof, ops.ATTN_PROFILE = ops.ATTN_PROFILE, None

        static_in = torch.empty_like(dev_imgs[0])
        graph = None
        if not args.no_graph:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                model(static_in.normal_())
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = model(static_in)

        def step(images):
            if graph is None:
                return model(images)
            static_in.copy_(images, non_blocking=True)
            graph.replay()
            return static_out

        for i in range(2):
            step(dev_imgs[i % n_bufs])
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        for i in range(args.steps):
            out = step(dev_imgs[i % n_bufs])
        e1.record()
        sync_all()
        clocks = sampler.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:                            # before the e2e replays overwrite static_out
            write_outputs(args.dump_outputs, step_outputs(out))
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        value = world * B * args.steps / (ms_total * 1e-3)

        # end to end: pinned host images -> H2D, logits -> host, every step
        host_imgs = [torch.randn(B, 3, c["img"], c["img"]).pin_memory() for _ in range(2)]
        host_out = torch.empty(B, c["classes"], dtype=torch.bfloat16).pin_memory()
        stage = [torch.empty_like(static_in) for _ in range(2)]
        copy_stream = torch.cuda.Stream()
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]

        def prefetch(i):
            k = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[k])
                stage[k].copy_(host_imgs[k], non_blocking=True)
                ready[k].record(copy_stream)

        for k in range(2):
            consumed[k].record()
        e2e_steps = args.steps
        sync_all()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        prefetch(0)
        for i in range(e2e_steps):
            if i + 1 < e2e_steps:
                prefetch(i + 1)
            k = i % 2
            torch.cuda.current_stream().wait_event(ready[k])
            out = step(stage[k])
            consumed[k].record()
            host_out.copy_(out, non_blocking=True)
            torch.cuda.current_stream().synchronize()                 # the caller consumes the logits every step
        t1.record()
        sync_all()
        tt = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * B * e2e_steps / (float(tt.item()) * 1e-3), "unit": "images/s", "h2d_bytes_per_step": img_bytes,
               "d2h_bytes_per_step": B * c["classes"] * 2, "steps": e2e_steps}

    peaks = load_peaks()

    def fam(prof, name):
        ms = sum(a.elapsed_time(b) for a, b, *_ in prof)
        fl = sum(r[-1] for r in prof)
        tf = fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        return {"kernel": name, "ms_per_step": ms / roof_steps, "launches_per_step": len(prof) / roof_steps,
                "achieved": tf, "frac": tf / peaks["tf_sustained"]}
    gem = fam(gprof, "gemm_bf16_kernel (tcgen05)")
    att = fam(aprof, "attn_fwd_kernel (tcgen05 flash attention)")
    dominant = att if att["ms_per_step"] > gem["ms_per_step"] else gem
    step_flops = fwd_flops_per_image(c) * B
    roofline = {"bound": "tensor", "kernel": dominant["kernel"], "achieved": dominant["achieved"], "peak": peaks["tf_sustained"],
                "unit": "TFLOP/s", "frac": dominant["frac"], "peak_source": peaks["source"] + " (sustained)", "traffic": None,
                "families": [gem, att],
                "timed_in": "eager replica of the forward (CUDA events around each launch) run before the timed region",
                "whole_step_tflops": step_flops / (ms_total / args.steps * 1e-3) / 1e12,
                "whole_step_frac_of_peak": step_flops / (ms_total / args.steps * 1e-3) / 1e12 / peaks["tf_sustained"]}
    pe_ms = sum(a.elapsed_time(b_) for a, b_, _, _ in pprof) / max(1, len(pprof))
    pe_bytes, pe_flops = (pprof[0][2], pprof[0][3]) if pprof else (0, 0)
    t_roof_ms = max(pe_bytes / (peaks["hbm_gbs"] * 1e9), pe_flops / (peaks["tf_sustained"] * 1e12)) * 1e3
    patch_embed = {"ms": pe_ms, "algorithmic_bytes": pe_bytes, "achieved_gbs": pe_bytes / (pe_ms * 1e-3) / 1e9 if pe_ms > 0 else 0.0,
                   "hbm_peak_gbs": peaks["hbm_gbs"], "frac_hbm": (pe_bytes / (pe_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if pe_ms > 0 else 0.0,
                   "frac_of_max_hbm_tensor_roofline": t_roof_ms / pe_ms if pe_ms > 0 else 0.0, "input_dtype": "fp32"}
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ips, sec, threads, cb = cpu_reference_forward(c, 2, 1, args.cpu_batch)
        cpu_baseline = {"value": ips, "unit": "images/s", "cores": threads, "kind": "port",
                        "sample": f"2 timed forwards (+1 warm-up) of batch {cb}, fp32, {threads} threads, same model"}
    if rank == 0:
        print(json.dumps({
            "metric": metric_name(args.config, args.curve, True), "value": value, "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.config} {args.curve} tokens, inference forward (eval, no_grad)", "batch_per_gpu": B,
                       "global_batch": B * world, "tokens": N, "params_dtype": "bf16", "parallelism": f"replicas x{world}",
                       "launch": "eager" if graph is None else "forward replayed from one CUDA graph",
                       "l2_policy": f"{n_bufs} rotating input batches of {img_bytes / 1e6:.0f} MB (together > L2)"},
            "roofline": roofline, "patch_embed": patch_embed, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step, "clocks": clocks}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def check_dp(c, device, rank, world, curve, overlap=False):
    """Data-parallel correctness on the hardware the scaling run uses (N > 1, default on): the SAME code path as the timed
    step — GraphedStep with FusedAdamW inside the graph, gradients written into the flat bucket, bucket ranges all-reduced
    on the side stream — on a depth-2 model of the config's width with dropout off and lr = 0, then rank 0 alone runs
    the full global batch eagerly. Asserts: mean of the ranks' first-step losses == full-batch loss, the all-reduced
    gradient / world == the full-batch gradient (norm and rel-L2, bf16 tolerance), identical buckets on every rank."""
    import torch.distributed as dist
    from src.training import distributed as D
    from src.training.graphs import GraphedStep
    from src.training.losses import SoftTargetCrossEntropy
    from src.training.optim import FusedAdamW
    cc = dict(c, depth=2)
    per = 8

    def build():
        m = build_b200_model(cc, device, curve)
        for mod in m.modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
            if isinstance(mod, torch.nn.MultiheadAttention):
                mod.dropout = 0.0
        return m
    g = torch.Generator(device=device).manual_seed(99)                # the same global batch on every rank
    x = torch.randn(per * world, 3, cc["img"], cc["img"], generator=g, device=device)
    la = torch.randint(0, cc["classes"], (per * world,), generator=g, device=device)
    tgt = soft_targets(la, la.roll(1), 0.3, cc["classes"])
    crit = SoftTargetCrossEntropy()
    model = build()
    D.sync_module(model)
    opt = FusedAdamW(model.parameters(), lr=0.0, weight_decay=0.0, max_grad_norm=1.0, overlap=overlap, comm_buckets=4 if overlap else 1)
    xs, ts = D.shard(x, rank, world), D.shard(tgt, rank, world)
    step = GraphedStep(model, crit, xs, ts, optimizer=opt)
    loss = step(xs, ts).detach().float().clone()
    torch.cuda.synchronize()
    g_dp = torch.cat([fb["g"].float() for fb in opt._flat]) / world
    overlapped, buckets = opt.last_overlapped_buckets, opt.last_num_buckets
    dist.all_reduce(loss, op=dist.ReduceOp.SUM)
    loss_dp = float(loss) / world
    lo, hi = g_dp.clone(), g_dp.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    same = bool(torch.equal(lo, hi))
    res = None
    if rank == 0:
        ref = build()
        ref.load_state_dict(model.state_dict())
        lf = crit(ref(x), tgt)
        lf.backward()
        names = [n for n, p in model.named_parameters() if p.requires_grad]
        gref = dict(ref.named_parameters())
        parts = []
        for fb in opt._flat:
            buf = torch.zeros(fb["n"], dtype=torch.float32, device=device)
            byid = {id(p): n for n, p in model.named_parameters()}
            for (p, off, k) in fb["views"]:
                gr = gref[byid[id(p)]].grad
                if gr is not None:
                    buf[off:off + k] = gr.float().reshape(-1)
            parts.append(buf)
        g_full = torch.cat(parts)
        rel = float((g_dp - g_full).norm() / g_full.norm())
        res = {"world": world, "global_batch": per * world, "loss_dp_mean": loss_dp, "loss_full_batch": float(lf),
               "grad_norm_dp": float(g_dp.norm()), "grad_norm_full_batch": float(g_full.norm()), "grad_rel_l2": rel,
               "buckets_identical_on_all_ranks": same, "allreduce_ranges": buckets, "ranges_overlapped_with_backward": overlapped}
        ok = (abs(loss_dp - float(lf)) < 2e-3 * max(1.0, abs(float(lf))) and rel < 3e-2 and same
              and abs(res["grad_norm_dp"] - res["grad_norm_full_batch"]) < 2e-2 * res["grad_norm_full_batch"])
        res["ok"] = bool(ok)
    flag = torch.tensor([1.0 if (res is None or res["ok"]) else 0.0], device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    opt.close()
    del step, opt, model
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    if float(flag) == 0.0:
        if rank == 0:
            print(json.dumps({"dp_check": res}), flush=True)
        raise SystemExit("bench.py: data-parallel check FAILED (sharded step != full-batch step)")
    return res


def cpu_reference_forward(c, steps, warmup, batch):
    """Forward of the CPU oracle port (stock torch fp32), all host threads; the batch shrinks for long sequences."""
    torch.set_num_threads(os.cpu_count() or 1)
    N = (c["img"] // c["patch"]) ** 2
    batch = max(1, min(batch, 16 * 196 // N)) if N > 196 else batch
    model = build_oracle_model(c).eval()
    x = torch.randn(batch, 3, c["img"], c["img"], generator=torch.Generator().manual_seed(0))
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            model(x)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return batch / sec, sec, torch.get_num_threads(), batch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch-gpu"])
    ap.add_argument("--config", default="vit_b16_224", choices=sorted(CONFIGS))
    ap.add_argument("--mode", default="train", choices=["train", "infer"],
                    help="train = the headline metric (fwd+bwd+optimizer); infer = forward only (BASELINE.json configs[1], [4])")
    ap.add_argument("--curve", default="hilbert", choices=["hilbert", "morton", "peano", "moore", "raster"],
                    help="token order (BASELINE.json config 3: Hilbert vs Morton vs raster); the headline metric is hilbert")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: config)")
    ap.add_argument("--cpu-batch", type=int, default=16, help="batch of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dropout", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--check-dp", dest="check_dp", action="store_true", default=None,
                    help="N > 1: assert the sharded step equals the full-batch step before timing (default: on when N > 1)")
    ap.add_argument("--no-check-dp", dest="check_dp", action="store_false")
    ap.add_argument("--overlap", action="store_true",
                    help="N > 1: all-reduce 4 bucket ranges on a side stream DURING backward instead of one all-reduce after it. Measured "
                         "slower (profiles/r2_bench_2gpu_*.json: 32.86 vs 32.49 ms, exposed 1.02 vs 0.61 ms): the persistent "
                         "one-CTA-per-SM kernels leave NCCL no SM to run on, and its CTAs then delay the next kernel's wave")
    ap.add_argument("--no-exposed", action="store_true", help="N > 1: skip the second (collective-free) capture that measures allreduce_exposed_ms")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32): logits, and for --mode train "
                         "also loss, params and grads; arrays above 4 Mi elements are a fixed seeded sample. Inputs are "
                         "seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    c = dict(CONFIGS[args.config])
    if args.config == "vit_b16_1024":
        args.mode = "infer"                                           # 4096-token config is an inference sweep
    if args.impl == "reference":
        return run_reference_arm(args, c)
    if args.impl == "torch-gpu":
        return run_torch_gpu_arm(args, c)
    if args.warmup < 3:
        args.warmup = 3
    if args.mode == "infer":
        return run_infer(args, c)

    import torch.distributed as dist
    from sfcvit import ops
    from src.training import distributed as D
    from src.training.losses import SoftTargetCrossEntropy
    from src.training.optim import FusedAdamW

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (B200); there is no CPU fallback")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    rank, world = D.init_from_env("nccl")
    B = args.batch or c["batch"]
    classes = c["classes"]

    dp_check = None
    if world > 1 and args.check_dp is not False:
        dp_check = check_dp(c, device, rank, world, args.curve, overlap=args.overlap)
    model = build_b200_model(c, device, args.curve)
    D.sync_module(model)
    if args.no_dropout:
        for m in model.modules():
            if isinstance(m, torch.nn.Dropout):
                m.p = 0.0
            if isinstance(m, torch.nn.MultiheadAttention):
                m.dropout = 0.0
    opt = FusedAdamW(model.parameters(), lr=3e-4, weight_decay=5e-5, max_grad_norm=1.0,   # main.py:288-289 + train.py:165
                     overlap=args.overlap, comm_buckets=4 if args.overlap else 1)
    crit = SoftTargetCrossEntropy()

    g = torch.Generator(device=device).manual_seed(1234 + rank)
    n_bufs = 4                                                        # distinct input batches: 4 x 154 MB > L2 (126 MB)
    dev_imgs = [torch.randn(B, 3, c["img"], c["img"], generator=g, device=device) for _ in range(n_bufs)]
    la = torch.randint(0, classes, (B,), generator=g, device=device)
    lb = torch.randint(0, classes, (B,), generator=g, device=device)
    tgt = soft_targets(la, lb, 0.3, classes)

    eager_logits = [None]                                             # detached: no autograd graph outlives the step

    def eager_step(images):
        opt.zero_grad(set_to_none=True)
        logits = model(images)
        eager_logits[0] = logits.detach()
        loss = crit(logits, tgt)
        loss.backward()
        opt.step()                                                    # all-reduce (N > 1) + clip + AdamW, fused
        return loss

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(args.warmup):                                      # eager warm-up (also builds the flat parameter buffers)
        eager_step(dev_imgs[i % n_bufs])
    sync_all()

    # ---------------- roofline pass: the same step launched eagerly with CUDA events around every GEMM launch
    ops.GEMM_PROFILE = []
    ops.PE_PROFILE = []
    roof_steps = min(3, max(1, args.steps))
    for i in range(roof_steps):
        eager_step(dev_imgs[i % n_bufs])
    sync_all()
    prof, ops.GEMM_PROFILE = ops.GEMM_PROFILE, None
    pe_prof, ops.PE_PROFILE = ops.PE_PROFILE, None
    gemm_ms = sum(a.elapsed_time(b) for a, b, _ in prof)
    gemm_flops = sum(f for _, _, f in prof)

    # ---------------- the step that is timed: forward + loss + backward + (bucketed NCCL all-reduce on a side stream,
    # N > 1) + grad-norm + clip + AdamW, ALL replayed from ONE CUDA graph; per step the host only hands lr / bias
    # corrections to the device (one 1-thread kernel) and replays
    graphed = None
    launches_per_step = None
    if not args.no_graph:
        from src.training.graphs import GraphedStep
        opt.zero_grad(set_to_none=True)
        loss = None                                                   # no live eager autograd graph during capture
        graphed = GraphedStep(model, crit, dev_imgs[0], tgt, optimizer=opt)
        launches_per_step = graphed.captured_launches + len(opt._flat)   # + the hyper-parameter store per flat buffer

    def step(images):
        if graphed is None:
            return eager_step(images)
        return graphed(images)

    for i in range(2):
        step(dev_imgs[i % n_bufs])
    sync_all()

    # ---------------- timed region 1: inputs resident in HBM
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for i in range(args.steps):
        loss = step(dev_imgs[i % n_bufs])
    e1.record()
    sync_all()
    ms_local = e0.elapsed_time(e1)
    launches = (ops.LAUNCHES - launches0) if graphed is None else launches_per_step * args.steps
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:                                # before the e2e steps train the model further
        logits = eager_logits[0] if graphed is None else graphed.logits
        write_outputs(args.dump_outputs, step_outputs(logits, loss, model))
    t = torch.tensor([ms_local], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * B * args.steps / (ms_total * 1e-3)

    peaks = load_peaks()
    gemm_tflops = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    step_flops = 3.0 * fwd_flops_per_image(c) * B
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")          # dram bytes per launch from the ncu --set full capture
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")      # IMPORTED from a committed ncu capture, not measured in this run
    roofline = {
        "bound": "tensor", "kernel": "gemm_bf16_kernel (tcgen05, all fwd/dgrad/wgrad launches)",
        "achieved": gemm_tflops, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
        "frac": gemm_tflops / peaks["tf_sustained"], "peak_source": peaks["source"] + " (sustained; kernels timed inside a long step)",
        "traffic": traffic, "traffic_source": "imported: profiles/gemm_traffic.json (ncu --set full capture of the same kernels, dram read+write per launch)",
        "launches_per_step": len(prof) / roof_steps,
        "avg_launch_ms": gemm_ms / max(1, len(prof)), "gemm_ms_per_step": gemm_ms / roof_steps,
        "timed_in": "eager replica of the step (same kernels, CUDA events around each launch) run just before the graph-replayed timed region",
        "whole_step_tflops": step_flops / (ms_total / args.steps * 1e-3) / 1e12,
        "whole_step_frac_of_peak": step_flops / (ms_total / args.steps * 1e-3) / 1e12 / peaks["tf_sustained"],
    }

    # second metric named by BASELINE.json: HBM GB/s of the fused curve-gather patch embed (algorithmic bytes = image read
    # once + token matrix written once, SURVEY.md §8d), timed in the same eager replica
    pe_ms = sum(a.elapsed_time(b_) for a, b_, _, _ in pe_prof) / max(1, len(pe_prof))
    pe_bytes = pe_prof[0][2] if pe_prof else 0
    pe_flops = pe_prof[0][3] if pe_prof else 0
    pe_gbs = pe_bytes / (pe_ms * 1e-3) / 1e9 if pe_ms > 0 else 0.0
    t_roof_ms = max(pe_bytes / (peaks["hbm_gbs"] * 1e9), pe_flops / (peaks["tf_sustained"] * 1e12)) * 1e3
    patch_embed = {"kernel": "patch_embed_tmem_kernel (curve-order gather written once into tensor memory, tcgen05 A-from-TMEM patch-embedding GEMM)", "ms": pe_ms,
                   "algorithmic_bytes": pe_bytes, "achieved_gbs": pe_gbs, "hbm_peak_gbs": peaks["hbm_gbs"],
                   "frac_hbm": pe_gbs / peaks["hbm_gbs"], "bound": "tensor at K = 768 (SURVEY.md §8d)",
                   "frac_of_max_hbm_tensor_roofline": t_roof_ms / pe_ms if pe_ms > 0 else 0.0, "input_dtype": "fp32"}

    # ---------------- timed region 2: end to end (pinned host inputs -> H2D every step, loss read back)
    host_imgs = [torch.randn(B, 3, c["img"], c["img"]).pin_memory() for _ in range(2)]
    stage = [torch.empty(B, 3, c["img"], c["img"], device=device) for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            stage[s].copy_(host_imgs[s], non_blocking=True)
            ready[s].record(copy_stream)

    for s in range(2):
        consumed[s].record()
    e2e_steps = args.steps
    sync_all()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    prefetch(0)
    loss_host = 0.0
    for i in range(e2e_steps):
        if i + 1 < e2e_steps:
            prefetch(i + 1)
        s = i % 2
        torch.cuda.current_stream().wait_event(ready[s])
        loss = step(stage[s])
        consumed[s].record()
        loss_host = float(loss.item())                                # device -> host read of the step's result
    t1.record()
    sync_all()
    tt = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_value = world * B * e2e_steps / (float(tt.item()) * 1e-3)
    e2e = {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": B * 3 * c["img"] * c["img"] * 4,
           "d2h_bytes_per_step": 4, "steps": e2e_steps, "last_loss": loss_host}

    # ---------------- N > 1: how much of the gradient all-reduce is NOT hidden behind backward: the same graph captured
    # again with the collectives left out (timing only; replicas diverge afterwards, so this is the last thing measured)
    allreduce_exposed_ms = None
    nocomm = None
    if world > 1 and graphed is not None and not args.no_exposed:
        from src.training.graphs import GraphedStep
        opt.skip_comm = True
        nocomm = GraphedStep(model, crit, dev_imgs[0], tgt, optimizer=opt)
        for i in range(2):
            nocomm(dev_imgs[i % n_bufs])
        sync_all()
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0.record()
        for i in range(args.steps):
            nocomm(dev_imgs[i % n_bufs])
        n1.record()
        sync_all()
        tn = torch.tensor([n0.elapsed_time(n1)], dtype=torch.float64, device=device)
        dist.all_reduce(tn, op=dist.ReduceOp.MAX)
        allreduce_exposed_ms = ms_total / args.steps - float(tn.item()) / args.steps
        opt.skip_comm = False

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ips, sec, threads = cpu_reference_throughput(c, 2, 1, args.cpu_batch)
        cpu_baseline = {"value": ips, "unit": "images/s", "cores": threads, "kind": "port",
                        "sample": f"2 timed steps (+1 warm-up) of batch {args.cpu_batch}, fp32, {threads} threads, same model/step as the GPU arm"}

    final_loss = float(loss.item())
    curve_gen = curve_generation_table(device) if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None
    pe_sweep = patch_embed_sweep(device, peaks) if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None
    torch_gpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            graphed = None                                            # free the captured activations first
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            ips, ms = torch_gpu_throughput(c, device, B, 3, 3, compiled=False)
            torch_gpu_baseline = {"value": ips, "unit": "images/s", "ms_per_step": ms, "variant": "eager, bf16 autocast, fused AdamW",
                                  "note": "stock torch modules on the same GPU (library kernels); `bench.py --impl torch-gpu` adds torch.compile"}
        except Exception as e:
            torch_gpu_baseline = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}

    if rank == 0:
        line = {
            "metric": metric_name(args.config, args.curve), "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.config} " + ("generalised-Hilbert (embed-and-prune)" if args.curve == "hilbert" else args.curve) + " tokens, training step fwd+bwd+clip+AdamW",
                       "batch_per_gpu": B, "global_batch": B * world, "tokens": (c["img"] // c["patch"]) ** 2,
                       "dropout": not args.no_dropout, "params_dtype": "bf16", "parallelism": f"dp{world}",
                       "launch": "eager" if graphed is None else "forward+backward+allreduce+clip+AdamW replayed from one CUDA graph",
                       "l2_policy": f"{n_bufs} rotating input batches of {B * 3 * c['img'] ** 2 * 4 / 1e6:.0f} MB (> 126 MB L2); activations per step ~GBs"},
            "roofline": roofline, "patch_embed": patch_embed, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": launches,
            "gpu_launches_per_step": launches / args.steps, "clocks": clocks, "loss": final_loss,
            "allreduce_buckets_per_step": opt.last_num_buckets, "allreduce_buckets_overlapped": opt.last_overlapped_buckets,
            "allreduce_exposed_ms": allreduce_exposed_ms, "dp_check": dp_check, "torch_gpu_baseline": torch_gpu_baseline,
            "curve_generation": curve_gen, "patch_embed_sweep": pe_sweep,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # captured graphs hold NCCL kernels: release them before the communicator goes away (destroying the process
        # group underneath live graphs hangs), then leave without the collective teardown
        graphed = nocomm = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
