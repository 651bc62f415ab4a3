"""The "library Blackwell path to beat" (SURVEY 8d): the UNMODIFIED reference model / loss / step
(oracle/_ref, see ref_loader.py) on device='cuda' -- torch's own kernels (cuBLASLt, cuDNN conv,
F.layer_norm, nn.GELU, nn.MultiheadAttention/SDPA, autograd, torch AdamW) under the flags of the
reference's GPU scripts (scripts/exp/gpu/*: --precision amp_bf16 --grad-checkpointing --local-loss
--gather-with-grad, TF32 + cudnn.benchmark as training/main.py:85-91).  A measurement, never on the
product path; none of clipa_b200's kernels run in it.
"""
from __future__ import annotations

import math


def library_baseline(wl: dict, batch: int, steps: int = 3, warmup: int = 2, grad_checkpointing: bool = True,
                     device: str = "cuda:0") -> dict:
    import torch
    from baseline.ref_loader import import_reference
    oc = import_reference()
    from training.precision import get_autocast            # training/precision.py:6-15
    dev = torch.device(device)
    torch.backends.cuda.matmul.allow_tf32 = True            # training/main.py:85-91
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.deterministic = False
    torch.manual_seed(0)
    model, _, _ = oc.create_model_and_transforms(wl["model"], precision="amp_bf16", device=dev,
                                                 force_image_size=wl["image"], pos_embed=wl["pos"],
                                                 output_dict=True)
    if grad_checkpointing:
        model.set_grad_checkpointing()
    model.train()
    named = list(model.named_parameters())
    exclude = lambda n, p: p.ndim < 2 or "bn" in n or "ln" in n or "bias" in n or "logit_scale" in n
    gain = [p for n, p in named if exclude(n, p) and p.requires_grad]
    rest = [p for n, p in named if not exclude(n, p) and p.requires_grad]
    opt = torch.optim.AdamW([{"params": gain, "weight_decay": 0.}, {"params": rest, "weight_decay": 0.2}],
                            lr=1.024e-3, betas=(0.9, 0.95), eps=1e-6)     # training/main.py:318-326
    loss_fn = oc.ClipLoss(local_loss=True, gather_with_grad=True, cache_labels=True, rank=0, world_size=1)
    autocast = get_autocast("amp_bf16")
    g = torch.Generator().manual_seed(1)
    images = torch.randn(batch, 3, wl["image"], wl["image"], generator=g).to(dev)
    ctx, vocab = model.context_length, model.vocab_size
    text = torch.randint(1, vocab - 1, (batch, ctx), generator=g)
    text[:, -1] = vocab - 1
    text = text.to(dev)

    def step():
        opt.zero_grad()
        with autocast():
            out = model(images, text)
            losses = loss_fn(**out, output_dict=True)
            total = sum(losses.values())
        total.backward()
        opt.step()
        with torch.no_grad():
            model.logit_scale.clamp_(0, math.log(100))
        return total

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    out = {"path": "unmodified reference (oracle/_ref) on torch CUDA library kernels, amp_bf16"
                   + (", grad checkpointing" if grad_checkpointing else ""),
           "model": wl["model"], "image_px": wl["image"], "batch": batch, "steps": steps, "warmup": warmup,
           "ms_per_step": ms, "pairs_per_s": batch / (ms * 1e-3), "loss": float(loss),
           "optimizer": "torch.optim.AdamW inside the timed step",
           "peak_hbm_gb": round(torch.cuda.max_memory_allocated(dev) / 2**30, 1)}
    if "gflop_per_pair" in wl:
        out["gflop_per_pair"] = wl["gflop_per_pair"]
    del model, opt, images, text
    torch.cuda.empty_cache()
    return out
