#!/usr/bin/env python
"""Headline benchmark: images/sec of the ViT-L 896x448 MIM training step (BASELINE.json configs[1]: bf16, batch 8
per GPU) through painter_b200, at N GPUs of one node (weak scaling: global batch 8*N, DDP over NCCL).

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference algorithm's CPU path (oracle port) on host cores

One step = forward + backward (+ DDP gradient all-reduce) + fused AdamW update on one synthetic batch.
`value` is timed with the batch already resident in HBM; `e2e` is the same step through the public module API with
the batch copied from pinned host memory and the loss read back every step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_IMAGE_TRAIN = 4769.23e9   # SURVEY.md section 8(d): forward 1589.74 GF, train = 3x
BATCH_PER_GPU = 8
H, W = 896, 448


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        return 1400.0, "fallback (B200_PROFILING.md sustained bf16)"


def _masks(B, seed, up=1):
    """BEiT block masks drawn by the reference MaskingGenerator (fixture made by oracle/make_golden.py); up = 2
    repeats every mask cell 2x2 for the 112x56 token grid of the 1792x896 workload."""
    import numpy as np
    import torch
    packed = torch.load(os.path.join(ROOT, "tests", "golden", "beit_masks_56x28.pt"), weights_only=False).numpy()
    m = np.unpackbits(packed, axis=-1)[..., :28]
    idx = [(seed * 7 + i) % m.shape[0] for i in range(B)]
    t = torch.from_numpy(m[idx].astype("int32"))
    if up > 1:
        t = t.repeat_interleave(up, 1).repeat_interleave(up, 2)
    return t


def _batch(B, seed, Hh=None, Ww=None):
    import torch
    Hh, Ww = Hh or H, Ww or W
    g = torch.Generator().manual_seed(1234 + seed)
    imgs = torch.randn(B, 3, Hh, Ww, generator=g)
    tgts = torch.randn(B, 3, Hh, Ww, generator=g)
    return imgs, tgts, _masks(B, seed, Hh // H), torch.ones(B, 3, Hh, Ww)


# BASELINE.json configs the bench can run: [1]/[3] "train" (the headline), [4] "long", [2] "seggpt" (run_seggpt)
WORKLOADS = {
    "train": dict(H=896, W=448, batch=8, flops=4769.23e9, tokens=1568,
                  name="ViT-L 896x448 bf16 MIM train step (fwd+bwd+AdamW), batch 8 per GPU "
                       "(BASELINE.json configs[1]; configs[3] at 8 GPUs)",
                  metric="images/sec ViT-L 896x448 MIM train step"),
    "long": dict(H=1792, W=896, batch=2, flops=28952.86e9, tokens=6272,
                 name="ViT-L 1792x896 long-sequence bf16 MIM train step (fwd+bwd+AdamW), 6272 tokens, batch 2 per GPU "
                      "(BASELINE.json configs[4])",
                 metric="images/sec ViT-L 1792x896 MIM train step"),
}
FLOPS_SEGGPT_FWD = 1589.74e9        # SURVEY.md section 8(d): SegGPT 1-prompt inference = one 896x448 forward


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_reference_step_time(threads, reps=1):
    """The reference's own CPU path: the UNMODIFIED `models_painter.painter_vit_large_patch16_input896x448_win_dec64_
    8glb_sl1()` module (staged copy under oracle/_ref, oracle/stage_reference.py; loaded through oracle/ref_loader)
    in torch-CPU eager fp32, train mode, B=1 896x448 forward + backward on `threads` host threads.  Falls back to the
    oracle port (kind "port") only if the staged tree is missing.  Returns (times of the `reps` steps, kind)."""
    import torch
    from oracle import painter_oracle as po
    from oracle import ref_loader
    from oracle.synth import synth_state_dict
    torch.set_num_threads(threads)
    cfg = po.PainterConfig()
    imgs, tgts, mask, valid = _batch(1, 0)
    times = []
    if ref_loader.available():
        kind = "reference"
        torch.manual_seed(0)
        model = ref_loader.models_painter().painter_vit_large_patch16_input896x448_win_dec64_8glb_sl1()
        model.load_state_dict(synth_state_dict(cfg, 0), strict=True)
        model.train()

        def one():
            for p in model.parameters():
                p.grad = None
            loss, _, _ = model(imgs, tgts, bool_masked_pos=mask, valid=valid.clone())
            loss.backward()
    else:
        kind = "port"
        sd = {k: v.requires_grad_(True) for k, v in synth_state_dict(cfg, 0).items()}

        def one():
            for v in sd.values():
                v.grad = None
            drops = po.draw_drop_scales(cfg, 1)
            loss, _, _ = po.forward(sd, cfg, imgs, tgts, mask, valid, drops=drops)
            loss.backward()
    for _ in range(reps):
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
    return times, kind


def reference_cuda_eager(dev, host, steps):
    """BASELINE.md section 3 "the practical bar to beat": the UNMODIFIED reference module in stock torch-CUDA eager on
    the same GPU - torch.autocast(bf16), same batch, forward + backward + torch's fused AdamW.  A labelled comparator
    next to the headline (the contract's reference arm stays the CPU path); baseline leg only, never on our path."""
    import torch
    from oracle import painter_oracle as po
    from oracle import ref_loader
    from oracle.synth import synth_state_dict
    if not ref_loader.available():
        return {"unavailable": "reference tree not staged (oracle/stage_reference.py)"}
    torch.cuda.empty_cache()
    model = ref_loader.models_painter().painter_vit_large_patch16_input896x448_win_dec64_8glb_sl1()
    model.load_state_dict(synth_state_dict(po.PainterConfig(), 0), strict=True)
    model = model.to(dev).train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.05, fused=True)
    batch = [t.to(dev) for t in host]

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss, _, _ = model(batch[0], batch[1], bool_masked_pos=batch[2], valid=batch[3].clone())
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    n = max(2, min(steps, 5))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        step()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / n
    peak_gb = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    del model, opt
    torch.cuda.empty_cache()
    return {"value": batch[0].shape[0] / (ms / 1e3), "unit": "images/s", "ms_per_step": ms, "steps": n,
            "what": "unmodified reference module, stock torch-CUDA eager (cuBLAS / cuDNN / ATen), torch.autocast(bf16), "
                    "same batch, fwd + bwd + torch fused AdamW, same GPU", "peak_mem_gib": round(peak_gb, 1)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = min(os.cpu_count() or 1, 32)   # beyond ~32 threads torch-CPU eager slows down (oversubscription)
    # one warm-up step, then --steps timed steps
    t, kind = cpu_reference_step_time(threads, reps=1 + args.steps)
    t = t[1:]
    ms = 1e3 * sum(t) / len(t)
    val = 1.0 / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "images/sec ViT-L 896x448 MIM train step", "value": val, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "ViT-L 896x448 MIM train step (fwd+bwd), B=1 per step on host cores",
                   "global_batch": 1, "parallelism": "cpu"},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": threads, "kind": kind,
                         "sample": f"{len(t)} x (B=1 train-mode forward+backward) of the "
                                   f"{'unmodified reference module' if kind == 'reference' else 'oracle port'}, "
                                   "torch-CPU eager fp32, after 1 warm-up"},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _seggpt_inputs(P=1, seed=0):
    """What seggpt_engine.inference_image hands to run_one_image: [P, 896, 448, 3] float64 ImageNet-normalised canvases
    (prompt over query; prompt target over a copy of itself)."""
    import numpy as np
    rng = np.random.RandomState(seed)
    mean, std = np.array([0.485, 0.456, 0.406]), np.array([0.229, 0.224, 0.225])
    img = (rng.rand(P, 896, 448, 3) - mean) / std
    half = (rng.rand(P, 448, 448, 3) > 0.5).astype(np.float64)
    tgt = (np.concatenate([half, half], axis=1) - mean) / std
    return img, tgt


def run_seggpt_reference(args):
    """--impl reference --workload seggpt: the unmodified reference SegGPT module driven by the unmodified
    seggpt_engine.run_one_image on the host cores (torch-CPU eager fp32)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    from oracle import painter_oracle as po
    from oracle import ref_loader
    from oracle.synth import synth_state_dict
    threads = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(threads)
    se = ref_loader.seggpt_engine()
    model = ref_loader.models_seggpt().seggpt_vit_large_patch16_input896x448()
    model.load_state_dict(synth_state_dict(po.PainterConfig(seggpt=True), 0), strict=True)
    model.eval()
    model.seg_type = "instance"
    img, tgt = _seggpt_inputs()
    times = []
    for _ in range(1 + args.steps):
        t0 = time.perf_counter()
        se.run_one_image(img, tgt, model, torch.device("cpu"))
        times.append(time.perf_counter() - t0)
    ms = 1e3 * sum(times[1:]) / len(times[1:])
    val = 1e3 / ms
    print(json.dumps({
        "impl": "reference", "metric": "images/sec SegGPT ViT-L in-context inference (1 prompt + 1 target 448x448)",
        "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": "SegGPT ViT-L run_one_image, 1 prompt pair + 1 target (BASELINE.json "
                                                    "configs[2]) on host cores", "parallelism": "cpu"},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": threads, "kind": "reference",
                         "sample": f"{len(times) - 1} x seggpt_engine.run_one_image (unmodified reference), torch-CPU "
                                   "eager fp32, after 1 warm-up"},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


def run_seggpt(args):
    """BASELINE.json configs[2]: SegGPT ViT-L in-context segmentation, 1 prompt pair + 1 target 448x448, 1 GPU.
    step = one forward of the stitched 896x448 canvases.  `value`: canvases resident in HBM, the forward replayed as
    ONE CUDA graph (painter_b200/graphs.py).  `e2e`: painter_b200.seggpt_engine.run_one_image - the reference entry
    point's signature - from host numpy arrays to the de-normalised result back on the host.  N > 1: independent
    replicas (inference shards by image; no collective), every rank runs the same loop."""
    if args.impl == "reference":
        return run_seggpt_reference(args)
    import numpy as np
    import torch
    import torch.distributed as dist
    from painter_b200 import _lib, dist_utils, models_seggpt, seggpt_engine
    from painter_b200.graphs import GraphedForward
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    model = models_seggpt.seggpt_vit_large_patch16_input896x448().to(dev).eval()
    with torch.no_grad():
        for n, p in model.named_parameters():
            if "rel_pos" in n:
                p.normal_(std=0.02)
    model.seg_type = "instance"
    img, tgt = _seggpt_inputs()
    steps, W_steps = args.steps, max(args.warmup, 3)
    x = torch.from_numpy(img).permute(0, 3, 1, 2).float().contiguous().to(dev)
    t = torch.from_numpy(tgt).permute(0, 3, 1, 2).float().contiguous().to(dev)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        sync()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        sync()
        return a.elapsed_time(b) / n

    # eager (one launch per kernel) for comparison, then the graph replay
    mask = seggpt_engine._half_mask(model, dev)
    valid = torch.ones_like(t)
    seg = torch.ones(1, 1, device=dev)

    def eager():
        with torch.no_grad():
            model(x, t, mask, valid, seg, -1)

    def measure(precision, n_graph):
        model.precision = precision
        for _ in range(W_steps):
            eager()
        n0 = _lib.launch_count()
        ms_eager = timed(eager, steps)
        launches = (_lib.launch_count() - n0) // steps
        gf = GraphedForward(model)
        for _ in range(W_steps):
            gf(x, t, mask, valid, seg, -1)
        ms_graph = timed(lambda: gf(x, t, mask, valid, seg, -1), n_graph)
        for _ in range(W_steps):
            seggpt_engine.run_one_image(img, tgt, model, dev)
        sync()
        t0 = time.perf_counter()
        for _ in range(steps):
            out = seggpt_engine.run_one_image(img, tgt, model, dev)
        torch.cuda.synchronize()
        ms_e2e = 1e3 * (time.perf_counter() - t0) / steps
        return ms_eager, ms_graph, ms_e2e, launches, out

    # fp32-accurate mode first (reported as an extra block), then the headline bf16 mode under the clock sampler
    acc = None
    if args.precision in ("both", "fp32"):
        a_eager, a_graph, a_e2e, a_launches, _ = measure("fp32", steps)
        acc = {"ms_per_step": a_graph, "value": world * 1e3 / a_graph, "eager_ms_per_step": a_eager,
               "e2e_ms_per_step": a_e2e, "e2e_value": world * 1e3 / a_e2e, "kernels_per_forward": int(a_launches),
               "note": "model.precision = 'fp32': split-bf16 (3 terms, 6 products) tensor-core GEMMs, fp32 softmax / "
                       "LayerNorm / exact-erf GELU; what precision='auto' selects for the reference's fp32 inference "
                       "calls (parity <= 1e-5, tests/test_gpu_accurate.py)"}
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms_eager, ms_graph, ms_e2e, launches, out = measure("bf16", steps)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)      # what run_one_image returned in the last timed e2e step
        np.save(os.path.join(args.dump_outputs, "result.npy"), out.numpy().astype(np.float64))
    ms_graph, ms_e2e, ms_eager = dist_utils.max_over_ranks([ms_graph, ms_e2e, ms_eager], device=dev)
    if rank == 0:
        peak, peak_src = _peaks()
        achieved = FLOPS_SEGGPT_FWD / (ms_graph / 1e3) / 1e12
        line = {
            "metric": "images/sec SegGPT ViT-L in-context inference (1 prompt + 1 target 448x448)",
            "value": world * 1e3 / ms_graph, "unit": "images/s", "n_gpus": world, "steps": steps, "warmup": W_steps,
            "ms_per_step": ms_graph, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": "SegGPT ViT-L in-context segmentation inference, 1 prompt pair + 1 target 448x448 "
                                   "(BASELINE.json configs[2]); replicas only when N > 1",
                       "parallelism": "single" if world == 1 else f"{world} replicas", "tokens_per_image": 1568,
                       "forward": "one CUDA-graph replay of the whole forward", "kernels_per_forward": int(launches),
                       "eager_ms_per_step": ms_eager,
                       "l2": "weights (0.74 GB bf16) exceed the 126 MB L2; no explicit flush"},
            "e2e": {"value": world * 1e3 / ms_e2e, "unit": "images/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": int(img.nbytes + tgt.nbytes), "d2h_bytes_per_step": int(out.numel() * 8),
                    "call": "painter_b200.seggpt_engine.run_one_image(img, tgt, model, device): numpy float64 canvases in, "
                            "de-normalised [448,448,3] float64 result on the host out (wall clock incl. both copies)"},
            "gpu_launches": int(launches) * steps,
            "roofline": {"bound": "tensor", "kernel": "whole forward (tcgen05 GEMMs + fused attention), one graph replay",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "peak_source": peak_src, "algorithmic_per_launch": FLOPS_SEGGPT_FWD, "traffic": None},
            "clocks": clk,
        }
        if acc is not None:
            line["fp32_accurate"] = acc
        if not args.no_cpu_baseline and world == 1:
            from oracle import painter_oracle as po  # noqa: F401  (checker / baseline leg only)
            import subprocess
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", "seggpt",
                                "--steps", "2"], capture_output=True, text=True)
            try:
                line["cpu_baseline"] = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception:
                line["cpu_baseline"] = {"error": (r.stderr or r.stdout)[-300:]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_PARAM_SAMPLES = 1024            # per parameter tensor, at positions seeded by the tensor's index
DUMP_PRED_MAX = 8 * 1568 * 768        # logits values written whole (the headline batch); a seeded sample beyond that


def dump_outputs(out_dir, loss, pred, mask, model):
    """What one training step hands back to its caller, as float32 .npy files (about 40 MB at the headline batch):
    loss.npy, pred.npy (the logits, [B, tokens, 768]), mask.npy and params_sample.npy, the parameters after the
    optimizer update at DUMP_PARAM_SAMPLES seeded positions per tensor (named_parameters() order)."""
    import numpy as np
    import torch
    from oracle.synth import sample_positions
    os.makedirs(out_dir, exist_ok=True)
    p = pred.detach().float()
    if p.numel() > DUMP_PRED_MAX:
        p = p.reshape(-1)[sample_positions(p.numel(), DUMP_PRED_MAX, 0).to(p.device)]
    params = [t.detach().reshape(-1)[sample_positions(t.numel(), DUMP_PARAM_SAMPLES, i).to(t.device)].float()
              for i, t in enumerate(model.parameters())]
    arrays = {"loss": loss.detach().float().reshape(1), "pred": p, "mask": mask.detach().float(),
              "params_sample": torch.cat(params)}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))


def main():
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line (NCCL prints its version banner there)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--bucket-mb", type=int, default=25, help="DDP gradient bucket size (N > 1)")
    ap.add_argument("--optimizer", default="pk", choices=["torch", "pk"],
                    help="AdamW implementation: painter_b200.optim.FusedAdamW (default) or torch's fused kernel")
    ap.add_argument("--dp", default="own", choices=["own", "ddp"],
                    help="N > 1: painter_b200.dist_utils.GradSync (bucketed all-reduce of the gradient arena issued "
                         "from backward; default) or stock DistributedDataParallel")
    ap.add_argument("--no-hi-prio", action="store_true",
                    help="N > 1: do NOT run the step on a high-priority CUDA stream (default: compute outranks NCCL's "
                         "stream, so a pending GEMM CTA gets a freed SM before a pending NCCL CTA does)")
    ap.add_argument("--bg-ctas", type=int, default=4,
                    help="N > 1, --dp own: CTA limit of the communicator used for all but the last gradient buckets")
    ap.add_argument("--sm-reserve", type=int, default=4,
                    help="N > 1, --dp own: SMs left to NCCL while gradient buckets are in flight")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--precision", default="both", choices=["bf16", "fp32", "both"],
                    help="seggpt workload: also time the fp32-accurate mode (reported under 'fp32_accurate')")
    ap.add_argument("--workload", default="train", choices=["train", "long", "seggpt"],
                    help="train = BASELINE configs[1]/[3] (headline), long = configs[4], seggpt = configs[2]")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graph", type=int, default=1,
                    help="1: the e2e step is painter_b200.train_utils.GraphedTrainStep (forward + backward + AdamW as one "
                         "CUDA-graph replay; N = 1 with the pk optimizer); 0: the reference loop's eager launches")
    ap.add_argument("--no-optimizer", action="store_true", help="diagnostic only; the reported step includes AdamW")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one computed as DIR/<name>.npy: train / long: "
                         "loss, logits, mask, a seeded sample of the updated parameters; seggpt: run_one_image's "
                         "result")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what painter_b200 computed; it has no meaning with --impl reference")
    if args.workload == "seggpt":
        return run_seggpt(args)
    if args.impl == "reference":
        return run_reference(args)
    wl = WORKLOADS[args.workload]
    if args.batch <= 0:
        args.batch = wl["batch"]

    import torch
    import torch.distributed as dist
    from painter_b200 import _lib, dist_utils, models_painter, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    W_steps = max(args.warmup, 3)
    B = args.batch
    if world > 1 and not args.no_hi_prio:
        torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=-1))

    torch.manual_seed(0)
    if args.workload == "long":
        from functools import partial
        model = models_painter.Painter(
            img_size=(1792, 896), patch_size=16, embed_dim=1024, depth=24, num_heads=16, drop_path_rate=0.1,
            window_size=14, qkv_bias=True, mlp_ratio=4, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6),
            window_block_indexes=(), residual_block_indexes=[], use_rel_pos=True, out_feature="last_feat",
            decoder_embed_dim=64, loss_func="smoothl1").to(dev)
    else:
        model = models_painter.painter_vit_large_patch16_input896x448_win_dec64_8glb_sl1().to(dev)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if "rel_pos" in n:
                p.normal_(std=0.02)
    model.train()
    net = model
    if world > 1:
        if args.dp == "own":
            gsync = dist_utils.GradSync(model, bucket_mb=args.bucket_mb if args.bucket_mb > 25 else 200,
                                        sm_reserve=args.sm_reserve, bg_ctas=args.bg_ctas)
        else:
            net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True,
                                                            bucket_cap_mb=args.bucket_mb)
    # the reference recipe (train_painter_vit_large.sh / main_train.py:344-348): AdamW over layer-decay groups
    from painter_b200.train_utils import adjust_learning_rate, param_groups_lrd
    groups = param_groups_lrd(model, 0.05, no_weight_decay_list=model.no_weight_decay(), layer_decay=0.8)
    if args.optimizer == "pk":
        from painter_b200.optim import FusedAdamW
        opt = FusedAdamW(groups, lr=1e-4, betas=(0.9, 0.999))
    else:
        opt = torch.optim.AdamW(groups, lr=1e-4, betas=(0.9, 0.999), fused=True)
    adjust_learning_rate(opt, 1.0, 1e-4, 0.0, 1, 15)

    host = [t.pin_memory() for t in _batch(B, dist_utils.rank_seed(0, rank) % 9973, wl["H"], wl["W"])]
    resident = [t.to(dev) for t in host]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host)

    # per-launch timing of the dominant kernel (the tcgen05 GEMM) with CUDA events on the launching stream
    gemm_log = []
    orig_gemm = ops.gemm
    record = {"on": False}

    def timed_gemm(a, b, *aa, **kw):
        if not record["on"]:
            return orig_gemm(a, b, *aa, **kw)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = orig_gemm(a, b, *aa, **kw)
        e1.record()
        M = a.shape[1] if kw.get("trans_a") else a.shape[0]
        K = a.shape[0] if kw.get("trans_a") else a.shape[1]
        N = b.shape[1] if kw.get("trans_b") else b.shape[0]
        gemm_log.append((2.0 * M * N * K, e0, e1, (M, N, K, int(bool(kw.get("trans_a"))),
                                                   int(bool(kw.get("trans_b"))), kw.get("kind", 0))))
        return out

    ops.gemm = timed_gemm
    import painter_b200.engine as eng
    eng.ops.gemm = timed_gemm

    def step(batch, read_loss):
        imgs, tgts, mask, valid = batch
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss, pred, bmask = net(imgs, tgts, bool_masked_pos=mask, valid=valid)
        loss.backward()
        if not args.no_optimizer:
            opt.step()
        opt.zero_grad(set_to_none=True)
        return loss.item() if read_loss else (loss, pred, bmask)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # End to end the step runs the way a user of painter_b200 runs it: train_utils.GraphedTrainStep = the same
    # forward + backward + AdamW captured once and replayed as ONE CUDA graph per iteration (single GPU, FusedAdamW).
    # The device-resident region below stays eager - its GEMM launches carry CUDA events - and so does the reference
    # loop reported next to the e2e figure.  (Measured: the replay is worth 0.5-0.8 % here; the eager step is already
    # GPU-bound, its ~2.7 us kernel boundaries are not launch latency - profiles/r02_step_timeline_warm.txt.)
    gstep = None
    if args.graph and world == 1 and args.optimizer == "pk" and not args.no_optimizer:
        from painter_b200.train_utils import GraphedTrainStep
        gstep = GraphedTrainStep(model, opt)

    for _ in range(W_steps):
        step(resident, False)
    sync()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    # ---------------- timed region 1: device-resident inputs ----------------
    # The per-launch CUDA events around the GEMMs live inside the timed region, but on two of its steps only (the
    # first and the middle one): ~340 event pairs per step cost ~1.6 ms of stream bubbles (scripts/step_timeline.py:
    # 62.6 ms per step without them against 64.2 ms with events on every step).
    sampled = {0, args.steps // 2}
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    for i in range(args.steps):
        record["on"] = i in sampled
        last = step(resident, False)
    e1.record()
    sync()
    launches = _lib.launch_count() - n0
    record["on"] = False
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last, model)
    del last
    # ---------------- timed region 2: end to end through the public API, the reference loop's way ----------------
    # strict = engine_train.train_one_epoch verbatim (engine_train.py:52-93): every step copies its batch from pinned
    # host memory with .to(device, non_blocking=True) on the compute stream, calls the module under autocast, reads
    # the loss with loss.item(), runs backward + the optimizer step and ends with torch.cuda.synchronize().
    # pipelined = the same work with painter_b200.data_utils.DevicePrefetcher issuing the copies one step ahead on a
    # side stream and each step's loss read back one step later (no per-step drain) - reported next to it.
    from painter_b200.data_utils import DevicePrefetcher

    def run_e2e(strict, n):
        seen = []
        losses = torch.empty(max(n, 1), dtype=torch.float32).pin_memory()
        sync()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        prev = None
        src = ([t.to(dev, non_blocking=True) for t in host] for _ in range(n)) if strict else \
            DevicePrefetcher((host for _ in range(n)), dev)
        for i, batch in enumerate(src):
            imgs, tgts, mask, valid = batch
            with torch.autocast("cuda", dtype=torch.bfloat16):
                loss, _, _ = net(imgs, tgts, bool_masked_pos=mask, valid=valid)
            if strict:
                seen.append(loss.item())                      # engine_train.py:68
            loss.backward()
            if not args.no_optimizer:
                opt.step()
            opt.zero_grad(set_to_none=True)
            if strict:
                torch.cuda.synchronize()                      # engine_train.py:93
            else:
                losses[i:i + 1].copy_(loss.detach().reshape(1), non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
                if prev is not None:
                    prev[1].synchronize()
                    seen.append(float(losses[prev[0]]))
                prev = (i, ev)
        if prev is not None:
            prev[1].synchronize()
            seen.append(float(losses[prev[0]]))
        b.record()
        sync()
        return a.elapsed_time(b), seen

    def run_e2e_graph(n):
        """The same iteration through the graphed public API: pinned-host batch copied into the step's static device
        buffers, one graph replay, loss.item() and torch.cuda.synchronize() every step."""
        seen = []
        sync()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            loss = gstep(*host)
            seen.append(loss.item())
            torch.cuda.synchronize()
        b.record()
        sync()
        return a.elapsed_time(b), seen

    run_e2e(True, 2)        # untimed: first-use costs of the loop (stream / buffer creation) are not steady state
    run_e2e(False, 2)
    ms_e2e, seen = run_e2e(True, args.steps)
    ms_e2e_pipe, _ = run_e2e(False, args.steps)
    last_loss = seen[-1]
    ms_e2e_eager = ms_e2e
    if gstep is not None:
        run_e2e_graph(2)
        ms_e2e, seen_g = run_e2e_graph(args.steps)
        last_loss = seen_g[-1]
    clk = clocks.stop() if rank == 0 else None

    ms_total, ms_e2e, ms_e2e_pipe = dist_utils.max_over_ranks([ms_total, ms_e2e, ms_e2e_pipe], device=dev)
    ms_step = ms_total / args.steps
    value = world * B / (ms_step / 1e3)
    e2e_val = world * B / (ms_e2e / args.steps / 1e3)

    if rank == 0:
        flops = sum(g[0] for g in gemm_log)
        gms = sum(g[1].elapsed_time(g[2]) for g in gemm_log)
        if os.environ.get("PK_BENCH_DETAIL"):      # per-shape GEMM table on stderr (diagnostics only)
            agg = {}
            for f, a, b, key in gemm_log:
                t = agg.setdefault(key, [0, 0.0, 0.0])
                t[0] += 1
                t[1] += a.elapsed_time(b)
                t[2] += f
            for key, (n, t, f) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                print(f"[gemm] M,N,K,tA,tB,kind={key} n/step={n / len(sampled):.0f} ms/step={t / len(sampled):.3f} "
                      f"TF/s={f / t / 1e9:.0f}", file=sys.stderr)
        peak, peak_src = _peaks()
        achieved = flops / (gms / 1e3) / 1e12 if gms > 0 else 0.0
        traffic = None      # DRAM bytes per launch of the GEMM kernel, from the committed ncu --set full capture
        for name in ("r02_ncu_gemm_traffic.json", "r01_ncu_gemm_traffic.json"):
            try:
                with open(os.path.join(ROOT, "profiles", name)) as f:
                    traffic = json.load(f)["avg_dram_bytes_per_launch"]
                break
            except (OSError, KeyError, ValueError):
                continue
        line = {
            "metric": wl["metric"], "value": value, "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": W_steps, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": wl["name"],
                       "global_batch": world * B, "parallelism": f"dp{world}" if world > 1 else "single",
                       "tokens_per_image": wl["tokens"],
                       "launch": "value: eager kernel launches (programmatic dependent launch between the hot kernels); "
                                 "e2e: " + ("one CUDA-graph replay per step (train_utils.GraphedTrainStep)"
                                            if gstep is not None else "eager"),
                       "optimizer": "none" if args.no_optimizer else (
                           "AdamW over lr_decay.param_groups_lrd groups (layer_decay 0.8, wd 0.05): " +
                           ("painter_b200.optim.FusedAdamW" if args.optimizer == "pk" else "torch fused AdamW")),
                       "data_parallel": "single" if world == 1 else (
                           "painter_b200.dist_utils.GradSync (arena buckets, NCCL all-reduce from backward)"
                           if args.dp == "own" else "torch DistributedDataParallel"),
                       "l2": "per-step working set (1.5 GB weights + >10 GB activations) far exceeds the 126 MB L2; "
                             "no explicit flush"},
            "e2e": {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps,
                    "loop": ("train_utils.GraphedTrainStep(model, optimizer)(pinned-host batch): copies into the step's "
                             "static device buffers, one CUDA-graph replay (forward + backward + AdamW), loss.item() "
                             "and torch.cuda.synchronize() every step") if gstep is not None else
                            "engine_train.train_one_epoch's (engine_train.py:52-93): pinned-host batch .to(device, "
                            "non_blocking=True) on the compute stream, loss.item() and torch.cuda.synchronize() every step",
                    "reference_loop_value": world * B / (ms_e2e_eager / args.steps / 1e3),
                    "reference_loop_note": "engine_train.train_one_epoch's loop verbatim (eager launches, .to(device), "
                                           "loss.item(), synchronize) driving the painter_b200 module",
                    "pipelined_value": world * B / (ms_e2e_pipe / args.steps / 1e3),
                    "pipelined_note": "same work with data_utils.DevicePrefetcher (copies one step ahead on a side "
                                      "stream) and each step's loss read back one step later (no per-step drain)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "pk::gemm_bf16_kernel (tcgen05 GEMM, all linear layers fwd/bwd)",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak if peak else None, "peak_source": peak_src,
                         "launches": len(gemm_log), "share_of_step": gms / (ms_step * len(sampled)), "traffic": traffic,
                         "algorithmic_per_launch": flops / max(len(gemm_log), 1),
                         "step_mfu": value / world * wl["flops"] / 1e12 / peak},
            "clocks": clk, "loss": last_loss,
        }
        if world == 1 and not args.no_cpu_baseline and args.workload == "train":
            try:
                line["reference_cuda_eager"] = reference_cuda_eager(dev, host, args.steps)
            except Exception as ex:      # a labelled extra: never let it take the bench line down
                line["reference_cuda_eager"] = {"error": repr(ex)[:200]}
            threads = min(os.cpu_count() or 1, 32)
            ts, kind = cpu_reference_step_time(threads, reps=2)
            line["cpu_baseline"] = {"value": 1.0 / ts[-1], "unit": "images/s", "cores": threads, "kind": kind,
                                    "sample": "1 x (B=1 train-mode forward+backward) of the unmodified reference "
                                              "module, torch-CPU eager fp32, after 1 warm-up"
                                    if kind == "reference" else
                                    "1 x (B=1 forward+backward) of the oracle port, torch-CPU fp32"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
