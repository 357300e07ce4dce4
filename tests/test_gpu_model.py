"""GPU parity of the painter_b200 modules against (i) golden vectors produced by the UNMODIFIED reference and
(ii) the CPU oracle.  Tolerances (bf16 tensor-core operands, fp32 accumulate; SURVEY.md section 8c calibration:
the reference's own bf16-vs-fp32 noise is loss 4e-7, logits RMS 9.5e-3 / max 1.3e-2, grads RMS 1.1e-2):
   loss   rel <= 1e-3 (north star)     logits  rms-rel <= 1.5e-2, max-rel <= 4e-2
   grads  rms-rel <= 1.5 x the reference's own bf16-autocast error on the same inputs, per tensor (SURVEY 8c); the
          fixed 4e-2 bound is only used where no noise measurement is available.
The same protocol at the benchmarked shapes, against the live reference, is in tests/test_gpu_fullsize.py.
"""
import pytest
import torch

from oracle import painter_oracle as po
from oracle.synth import synth_inputs, synth_state_dict

from _common import build_model, load_golden, rel_max, rel_rms, sampled_rms_rel

pytestmark = pytest.mark.gpu

LOSS_TOL, LOGIT_RMS, LOGIT_MAX, GRAD_RMS = 1e-3, 1.5e-2, 4e-2, 4e-2
NOISE_RATIO = 1.5


def _to(dev, *ts):
    return [t.to(dev) for t in ts]


def _reference_bf16_noise(cfg, sd, imgs, tgts, mask, valid, drops=None):
    """Error of the reference algorithm ITSELF when run under torch.autocast('cuda', bf16) (the oracle restatement
    uses the same torch ops, so CUDA autocast gives it the reference's dtype flow) against its fp32 result.
    SURVEY.md section 8(c): ours must stay within 1.5x of this noise floor."""
    sdc = {k: v.cuda().requires_grad_(True) for k, v in sd.items()}
    args = [t.cuda() for t in (imgs, tgts, mask, valid)]
    d = None if drops is None else [tuple(t.cuda() for t in pair) for pair in drops]
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss, pred, _ = po.forward(sdc, cfg, *args, drops=d)
    loss.float().backward()
    return {k: v.grad for k, v in sdc.items()}, pred.float()


def _check_grads(model, ref_grads, ref_norms=None, noise=None):
    named = dict(model.named_parameters())
    bad = []
    for k, g in ref_grads.items():
        err = (lambda a: sampled_rms_rel(a, g)) if isinstance(g, dict) else (lambda a: rel_rms(a, g))  # seeded sample
        e = err(named[k].grad)
        tol = GRAD_RMS if noise is None else NOISE_RATIO * err(noise[k])
        if e > tol:
            bad.append((k, e, tol))
    if ref_norms is not None:
        for k, n in ref_norms.items():
            gn = named[k].grad.float().norm().item()
            if abs(gn - n) > 0.05 * max(n, 1e-5) + 1e-6:
                bad.append((k + "(norm)", gn, n))
    assert not bad, bad[:10]


def test_painter_tiny_eval_fwd_bwd_vs_reference_golden():
    gold = load_golden("painter_tiny.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    model, _ = build_model(cfg, gold["weight_seed"])
    model.eval()
    imgs, tgts, mask, valid = _to("cuda", *synth_inputs(cfg, **gold["inputs"]))
    loss, pred, m = model(imgs, tgts, mask, valid)
    ev = gold["eval"]
    assert abs(loss.item() - ev["loss"].item()) <= LOSS_TOL * abs(ev["loss"].item())
    assert rel_rms(pred, ev["pred"]) <= LOGIT_RMS and rel_max(pred, ev["pred"]) <= LOGIT_MAX
    assert torch.equal(m.cpu(), ev["mask"])
    loss.backward()
    noise, npred = _reference_bf16_noise(cfg, synth_state_dict(cfg, gold["weight_seed"]), imgs, tgts, mask, valid)
    print("pred rms-rel ours", rel_rms(pred, ev["pred"]), "reference-bf16", rel_rms(npred, ev["pred"]))
    _check_grads(model, ev["grads"], ev["grad_norms"], noise)


def test_painter_tiny_train_mode_droppath_replay():
    gold = load_golden("painter_tiny.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    model, _ = build_model(cfg, gold["weight_seed"])
    model.train()
    imgs, tgts, mask, valid = _to("cuda", *synth_inputs(cfg, **gold["inputs"]))
    torch.manual_seed(gold["train_seed"])
    drops = po.draw_drop_scales(cfg, imgs.shape[0])  # the reference's CPU draws, replayed
    model._drop_scales = lambda i, Bp, dev: tuple(t.to(dev) for t in drops[i])
    loss, pred, _ = model(imgs, tgts, mask, valid)
    tr = load_golden("painter_tiny_train.pt")
    assert abs(loss.item() - tr["loss"].item()) <= LOSS_TOL * abs(tr["loss"].item())
    assert rel_rms(pred, tr["pred"]) <= LOGIT_RMS
    loss.backward()
    noise, _ = _reference_bf16_noise(cfg, synth_state_dict(cfg, gold["weight_seed"]), imgs, tgts, mask, valid, drops)
    _check_grads(model, tr["grads"], tr["grad_norms"], noise)


def test_painter_tiny_interpolated_tables():
    """64x32 input on the 128x64 model: abs-pos bicubic + rel-pos linear resize (vitdet_utils.py:75-86,141-153)."""
    gold = load_golden("painter_tiny.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    model, _ = build_model(cfg, gold["weight_seed"])
    model.eval()
    it = gold["interp"]
    i2, t2, mk2, v2 = _to("cuda", *synth_inputs(cfg, **it["inputs"]))
    with torch.no_grad():
        loss, pred, _ = model(i2, t2, mk2, v2)
    assert abs(loss.item() - it["loss"].item()) <= LOSS_TOL * abs(it["loss"].item())
    assert rel_rms(pred, it["pred"]) <= LOGIT_RMS


def test_painter_tiny_window_blocks_vs_reference_golden():
    """Real windowed blocks (non-stock, parameterised): ws=7 on the 8x4 grid pads to 14x7 (vitdet_utils.py:29-33)."""
    gold = load_golden("painter_tiny_window.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    model, _ = build_model(cfg, gold["weight_seed"])
    model.eval()
    assert sorted({b.window_size for b in model.blocks}) == [0, 7]
    imgs, tgts, mask, valid = _to("cuda", *synth_inputs(cfg, **gold["inputs"]))
    loss, pred, _ = model(imgs, tgts, mask, valid)
    ev = gold["eval"]
    assert abs(loss.item() - ev["loss"].item()) <= LOSS_TOL * abs(ev["loss"].item())
    assert rel_rms(pred, ev["pred"]) <= LOGIT_RMS
    loss.backward()
    noise, _ = _reference_bf16_noise(cfg, synth_state_dict(cfg, gold["weight_seed"]), imgs, tgts, mask, valid)
    _check_grads(model, ev["grads"], ev["grad_norms"], noise)


def test_seggpt_tiny_prompts_and_ensemble():
    gold = load_golden("seggpt_tiny.pt")
    cfg = po.PainterConfig(**gold["cfg"])
    model, _ = build_model(cfg, gold["weight_seed"])
    model.eval()
    h, w = cfg.grid
    for c in gold["cases"]:
        x, t, _, _ = synth_inputs(cfg, c["P"], c["seed"])
        bm = torch.zeros(1, h * w)
        bm[:, h * w // 2:] = 1
        seg = torch.full((c["P"], 1), float(c["seg_type"]))
        with torch.no_grad():
            loss, pred, _ = model(x.cuda(), t.cuda(), bm.cuda(), torch.ones_like(t).cuda(), seg.cuda(),
                                  c["merge_between_batch"])
        assert abs(loss.item() - c["loss"].item()) <= LOSS_TOL * abs(c["loss"].item()), c["P"]
        assert rel_rms(pred, c["pred"]) <= LOGIT_RMS, c["P"]


def test_full_size_forward_vs_oracle():
    """ViT-L 896x448, B=1, eval forward against the CPU oracle (fp32) on the same seeded weights/inputs."""
    cfg = po.PainterConfig()
    model, sd = build_model(cfg, 1)
    model.eval()
    imgs, tgts, mask, valid = synth_inputs(cfg, 1, 21)
    with torch.no_grad():
        loss, pred, _ = model(imgs.cuda(), tgts.cuda(), mask.cuda(), valid.cuda())
        torch.set_num_threads(min(32, torch.get_num_threads()))  # 100+ threads oversubscribe the CPU oracle
        rl, rp, _ = po.forward(sd, cfg, imgs, tgts, mask, valid)
    assert abs(loss.item() - rl.item()) <= LOSS_TOL * abs(rl.item())
    assert rel_rms(pred, rp) <= LOGIT_RMS and rel_max(pred, rp) <= LOGIT_MAX


def test_amp_gradscaler_training_steps_like_engine_train():
    """The step of engine_train.train_one_epoch (:56-93) + misc.NativeScalerWithGradNormCount (:252-269):
    fp16-autocast context, GradScaler, grad clipping, AdamW — must run and reduce the loss."""
    cfg = po.PainterConfig(img_size=(128, 64), embed_dim=128, num_heads=2, decoder_embed_dim=64)
    model, _ = build_model(cfg, 0)
    model.train()
    opt = torch.optim.AdamW(model.parameters(), lr=2e-4, betas=(0.9, 0.999), weight_decay=0.05)
    scaler = torch.cuda.amp.GradScaler()
    imgs, tgts, mask, valid = _to("cuda", *synth_inputs(cfg, 4, 3))
    losses = []
    for step in range(6):
        with torch.cuda.amp.autocast():
            loss, y, m = model(imgs, tgts, bool_masked_pos=mask, valid=valid)
        losses.append(loss.item())
        assert torch.isfinite(loss)
        scaler.scale(loss).backward()
        scaler.unscale_(opt)
        norm = torch.nn.utils.clip_grad_norm_(model.parameters(), 3.0)
        assert torch.isfinite(norm)
        scaler.step(opt)
        scaler.update()
        opt.zero_grad()
    assert losses[-1] < losses[0], losses


def test_no_cpu_fallback():
    cfg = po.PainterConfig(img_size=(128, 64), embed_dim=128, num_heads=2, decoder_embed_dim=64)
    from functools import partial
    from painter_b200 import models_painter
    m = models_painter.Painter(img_size=(128, 64), embed_dim=128, num_heads=2, decoder_embed_dim=64,
                               use_rel_pos=True, depth=24, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))
    x = torch.randn(1, 3, 128, 64)
    with pytest.raises(RuntimeError):
        m(x, x, torch.zeros(1, 8, 4), torch.ones(1, 3, 128, 64))


def test_device_prefetcher_yields_every_pinned_batch_once():
    """engine_train.py:52-56 moves each batch to the device at the top of the step; the prefetcher does the same
    copy one step ahead on a side stream."""
    from painter_b200.data_utils import DevicePrefetcher
    host = [(torch.full((64, 64), float(i)).pin_memory(), torch.arange(16).add(i).pin_memory()) for i in range(5)]
    seen = []
    for a, b in DevicePrefetcher(iter(host), "cuda"):
        assert a.is_cuda and b.is_cuda
        seen.append((a.sum().item(), b[0].item()))
    assert seen == [(64.0 * 64 * i, i) for i in range(5)]


def test_painter_tiny_other_loss_functions_vs_reference_golden():
    """loss_func in {l1, l2, l1l2} (models_painter.py:453-458; non-stock): forward loss and the gradients that flow
    through the fused decoder head, against vectors produced by the unmodified reference."""
    gold = load_golden("painter_tiny_losses.pt")
    for c in gold["cases"]:
        cfg = po.PainterConfig(**c["cfg"])
        model, sd = build_model(cfg, c["weight_seed"])
        model.eval()
        imgs, tgts, mask, valid = _to("cuda", *synth_inputs(cfg, **c["inputs"]))
        loss, _, _ = model(imgs, tgts, mask, valid)
        assert abs(loss.item() - c["loss"].item()) <= LOSS_TOL * abs(c["loss"].item()), cfg.loss_func
        loss.backward()
        noise, _ = _reference_bf16_noise(cfg, sd, imgs, tgts, mask, valid)
        _check_grads(model, c["grads"], c["grad_norms"], noise)


def test_fused_adamw_trains_the_gemm_weights():
    """ADVICE r1 (high): FusedAdamW writes parameters through raw pointers; the bf16 GEMM-weight cache of
    engine.bf16_weight must see every update (version bump) - the loss must fall and the cached bf16 copy must equal
    the fp32 master after each step."""
    from painter_b200 import engine
    from painter_b200.optim import FusedAdamW
    cfg = po.PainterConfig(img_size=(128, 64), embed_dim=128, num_heads=2, decoder_embed_dim=64)
    model, _ = build_model(cfg, 0)
    model.train()
    opt = FusedAdamW(model.parameters(), lr=2e-4, betas=(0.9, 0.999), weight_decay=0.05)
    imgs, tgts, mask, valid = _to("cuda", *synth_inputs(cfg, 4, 3))
    losses = []
    w = model.blocks[5].mlp.fc1.weight
    for step in range(6):
        loss, _, _ = model(imgs, tgts, bool_masked_pos=mask, valid=valid)
        losses.append(loss.item())
        loss.backward()
        before = w.detach().clone()
        opt.step()
        opt.zero_grad(set_to_none=True)
        assert not torch.equal(before, w.detach()), "parameter did not move"
        assert torch.equal(engine.bf16_weight(w), w.detach().bfloat16()), "stale bf16 weight cache after the step"
    assert losses[-1] < losses[0], losses


def test_graphed_train_step_equals_eager_steps():
    """train_utils.GraphedTrainStep: forward + backward + FusedAdamW as one CUDA-graph replay per iteration.  With
    DropPath off (eval-mode module, as the parity tests run it) every replay must reproduce the eager step: same
    losses, same parameters after 4 iterations with a learning rate that changes every iteration, and the warm-up
    iterations of the capture must leave no trace (parameters / optimizer state restored)."""
    from painter_b200.optim import FusedAdamW
    from painter_b200.train_utils import GraphedTrainStep
    cfg = po.PainterConfig(img_size=(128, 64), embed_dim=128, num_heads=2, decoder_embed_dim=64)
    model, _ = build_model(cfg, 0)
    twin, _ = build_model(cfg, 0)
    model.eval()
    twin.eval()
    batches = [_to("cuda", *synth_inputs(cfg, 4, 3 + i)) for i in range(4)]
    lrs = [2e-4, 1.5e-4, 1e-4, 0.5e-4]
    opt_e = FusedAdamW(twin.parameters(), lr=lrs[0], betas=(0.9, 0.999), weight_decay=0.05)
    eager = []
    for (imgs, tgts, mask, valid), lr in zip(batches, lrs):
        for g in opt_e.param_groups:
            g["lr"] = lr
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss, _, _ = twin(imgs, tgts, bool_masked_pos=mask, valid=valid)
        loss.backward()
        opt_e.step()
        opt_e.zero_grad(set_to_none=True)
        eager.append(loss.item())
    opt_g = FusedAdamW(model.parameters(), lr=lrs[0], betas=(0.9, 0.999), weight_decay=0.05)
    step = GraphedTrainStep(model, opt_g)
    graphed = []
    for (imgs, tgts, mask, valid), lr in zip(batches, lrs):
        for g in opt_g.param_groups:
            g["lr"] = lr
        graphed.append(step(imgs, tgts, mask, valid).item())
    assert len(step.entries) == 1
    # the first replay sees exactly the eager step's inputs and weights; later ones differ by the summation order of
    # the stream-K weight-gradient atomics (as two eager runs do): ~1e-5 relative on the loss after three updates
    assert abs(eager[0] - graphed[0]) <= 1e-6 * abs(eager[0]), (eager, graphed)
    for a, b in zip(eager, graphed):
        assert abs(a - b) <= 1e-4 * max(1.0, abs(a)), (eager, graphed)
    ref0, _ = build_model(cfg, 0)
    for (n, p), (_, q), (_, p0) in zip(model.named_parameters(), twin.named_parameters(), ref0.named_parameters()):
        if p.numel() < 4096:
            continue
        du_g, du_e = (p.detach() - p0.detach()).double(), (q.detach() - p0.detach()).double()
        rel = (du_g - du_e).norm().item() / (du_e.norm().item() + 1e-30)
        assert rel <= 0.1, (n, rel)       # four Adam updates agree to a few per cent in every large tensor
    st_g, st_e = opt_g.state[model.blocks[3].mlp.fc1.weight], opt_e.state[twin.blocks[3].mlp.fc1.weight]
    assert st_g["step"] == st_e["step"] == 4
    rel = (st_g["exp_avg_sq"].double() - st_e["exp_avg_sq"].double()).norm() / st_e["exp_avg_sq"].double().norm()
    # second moments after four updates: the two runs differ by the summation order of the stream-K weight-gradient
    # atomics (1.1e-3 measured between two otherwise identical runs on the B200), not by the captured optimizer step
    assert rel.item() <= 5e-3, rel.item()


def test_gradient_arena_views_accumulation_and_fused_step():
    """painter_b200/arena.py: p.grad is a view of the flat arena after a backward; a second backward without
    zero_grad accumulates (scratch slab) to exactly twice the gradient; FusedAdamW consumes and clears the arena and
    takes the same step as torch.optim.AdamW."""
    from painter_b200.arena import get_arena
    from painter_b200.optim import FusedAdamW, global_grad_norm
    cfg = po.PainterConfig(img_size=(128, 64), embed_dim=128, num_heads=2, decoder_embed_dim=64)
    model, _ = build_model(cfg, 0)
    twin, _ = build_model(cfg, 0)
    model.eval()
    twin.eval()
    imgs, tgts, mask, valid = _to("cuda", *synth_inputs(cfg, 2, 3, valid_kind="mixed"))
    loss, _, _ = model(imgs, tgts, mask, valid)
    loss.backward()
    arena = get_arena(model)
    assert arena.grads_in_arena()
    g1 = {n: p.grad.clone() for n, p in model.named_parameters()}
    n1 = global_grad_norm(model.parameters()).item()
    ref_norm = torch.sqrt(sum(g.double().pow(2).sum() for g in g1.values())).item()
    assert abs(n1 - ref_norm) <= 1e-5 * ref_norm
    loss, _, _ = model(imgs, tgts, mask, valid)
    loss.backward()                                         # accumulation: p.grad is live
    for n, p in model.named_parameters():
        assert rel_rms(p.grad, 2 * g1[n]) < 1e-5, n
    assert arena.grads_in_arena()
    # one optimizer step from the single-backward gradient, against torch.optim.AdamW on an identical twin
    for p in model.parameters():
        p.grad = None
    loss, _, _ = model(imgs, tgts, mask, valid)
    loss.backward()
    lt, _, _ = twin(imgs, tgts, mask, valid)
    lt.backward()
    opt = FusedAdamW(model.parameters(), lr=1e-3, betas=(0.9, 0.999), weight_decay=0.05)
    topt = torch.optim.AdamW(twin.parameters(), lr=1e-3, betas=(0.9, 0.999), weight_decay=0.05)
    opt.step()
    topt.step()
    torch.cuda.synchronize()
    assert arena.clean and float(arena.slab.abs().max()) == 0.0, "the fused step must leave the arena zeroed"
    worst = max(((p - q).abs().max() / q.abs().max().clamp_min(1e-12)).item()
                for p, q in zip(model.parameters(), twin.parameters()))
    # Adam's first step is lr * sign(g) wherever |g| >> eps: a sign flip of a ~0 gradient moves a weight by 2 lr
    assert worst < 5e-2, worst
    frac_same = sum(((p - q).abs() <= 1e-6 + 1e-4 * q.abs()).sum().item() for p, q in
                    zip(model.parameters(), twin.parameters())) / sum(p.numel() for p in model.parameters())
    assert frac_same > 0.98, frac_same
    opt.zero_grad(set_to_none=True)
    loss2, _, _ = model(imgs, tgts, mask, valid)            # next step runs on the kernel-refreshed bf16 operands
    loss2.backward()
    assert arena.grads_in_arena() and torch.isfinite(loss2)


def test_nccl_world2_gradsync_equals_mean_of_rank_gradients(tmp_path):
    """GradSync over NCCL on the CUDA module (needs 2 GPUs): the synchronised gradient of every parameter equals the
    mean of the two ranks' local gradients."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import subprocess
    import sys
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path / "nccl.json")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611",
                        os.path.join(root, "scripts", "nccl_gradsync_check.py"), out],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    import json
    res = json.load(open(out))
    assert res["max_rel_err"] < 1e-5, res
