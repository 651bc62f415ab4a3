"""Generates tests/golden/*.npz by running the UNMODIFIED reference (imported from oracle/_ref, installed by
oracle/install_reference.sh) on seeded synthetic weights and inputs, on the CPU.

The vectors it writes are committed; the tests read only those.  Usage:  python oracle/make_golden.py

What is pinned per case (fp32 reference run, plus a pure-bf16 run that calibrates the bf16
tolerance): image/text features, loss, and gradients of logit_scale, visual.proj, text_projection,
the first vision block's in_proj_weight and the token embedding rows that were used.
A 2-rank Gloo run pins ClipLoss(local_loss=True, gather_with_grad=True) loss and feature gradients.
"""
from __future__ import annotations

import importlib.machinery
import json
import os
import sys
import tempfile
from pathlib import Path
from unittest.mock import MagicMock

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle.weights import (BASELINE_DIM_BATCH, BASELINE_DIM_CASES, CONFIG1, TINY_CONFIGS, make_inputs,  # noqa: E402
                            make_state_dict)

REF = str(ROOT / "oracle" / "_ref")
GOLD = ROOT / "tests" / "golden"


def import_reference():
    """The tokenizer module imports ftfy/tensorflow(_text) unconditionally (open_clip/tokenizer.py:
    11,16-18); they are not on this path, so stub them."""
    for n in ("ftfy", "tensorflow", "tensorflow_text"):
        if n not in sys.modules:
            m = MagicMock()
            m.__spec__ = importlib.machinery.ModuleSpec(n, None)
            sys.modules[n] = m
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import open_clip  # noqa
    return open_clip


CASES = [
    # name, cfg, batch, image_size, pos_embed, seed
    ("tiny-cls", TINY_CONFIGS["tiny-cls"], 6, 64, "learnable", 11),
    ("tiny-gap-h80", TINY_CONFIGS["tiny-gap-h80"], 5, 48, "sin_cos_2d", 12),
    ("tiny-bigvision", TINY_CONFIGS["tiny-bigvision"], 4, 64, "learnable", 13),
    ("config1-vitb32", CONFIG1, 8, 192, "sin_cos_2d", 14),
]


def run_reference(open_clip, name, cfg, batch, image_size, pos_embed, seed, precision, compact=False):
    """precision: 'fp32' | 'bf16' (pure bf16 weights, open_clip/model.py:78-86) | 'amp_bf16' (fp32 master
    weights, forward + loss under bf16 autocast: training/precision.py:11-13 selects
    torch.cuda.amp.autocast(dtype=bfloat16) -- a no-op without CUDA, so the same context is opened for the CPU
    device, the closest same-mode run the reference can do in this container).
    compact: store 64x64 corners instead of whole projection gradients (BASELINE-dimension cases)."""
    tmp = Path(tempfile.mkdtemp())
    (tmp / f"golden-{name}.json").write_text(json.dumps(cfg))
    open_clip.add_model_config(tmp)
    model, _, _ = open_clip.create_model_and_transforms(
        f"golden-{name}", precision=precision, device="cpu", force_image_size=image_size,
        pos_embed=pos_embed, output_dict=True)
    sd = make_state_dict(cfg, seed, image_size=image_size, pos_embed=pos_embed)
    missing = model.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    model.train()
    images, text = make_inputs(cfg, batch, seed + 1000, image_size=image_size)
    if precision == "bf16":
        images = images.to(torch.bfloat16)
    import contextlib
    ctx = torch.autocast(device_type="cpu", dtype=torch.bfloat16) if precision == "amp_bf16" else contextlib.nullcontext()
    loss_fn = open_clip.ClipLoss()
    with ctx:
        out = model(images, text)
        loss = loss_fn(out["image_features"], out["text_features"], out["logit_scale"])
    for p in model.parameters():
        p.grad = None
    out["image_features"].retain_grad()
    out["text_features"].retain_grad()
    loss.backward()
    used = torch.unique(text)
    g = {k: v for k, v in model.named_parameters()}
    res = {
        "image_features": out["image_features"].detach().float().numpy(),
        "text_features": out["text_features"].detach().float().numpy(),
        "logit_scale": out["logit_scale"].detach().float().numpy(),
        "loss": loss.detach().float().numpy(),
        "loss_dtype": str(loss.dtype),
        "d_image_features": out["image_features"].grad.float().numpy(),
        "d_text_features": out["text_features"].grad.float().numpy(),
        "g_logit_scale": g["logit_scale"].grad.float().numpy(),
        "g_visual_proj": g["visual.proj"].grad.float().numpy()[:64, :64] if compact else g["visual.proj"].grad.float().numpy(),
        "g_text_projection": g["text_projection"].grad.float().numpy()[:64, :64] if compact else g["text_projection"].grad.float().numpy(),
        "g_visual_proj_norm": np.array(g["visual.proj"].grad.float().norm().item()),
        "g_v0_in_proj_weight": g["visual.transformer.resblocks.0.attn.in_proj_weight"].grad.float().numpy()[:64, :64],
        "g_v0_in_proj_bias": g["visual.transformer.resblocks.0.attn.in_proj_bias"].grad.float().numpy(),
        "g_vlast_c_fc_bias": g[f"visual.transformer.resblocks.{cfg['vision_cfg']['layers'] - 1}.mlp.c_fc.bias"].grad.float().numpy(),
        "g_t0_ln_1_weight": g["transformer.resblocks.0.ln_1.weight"].grad.float().numpy(),
        "g_class_embedding": g["visual.class_embedding"].grad.float().numpy(),
        "g_conv1_norm": np.array(g["visual.conv1.weight"].grad.float().norm().item()),
        "g_token_rows": g["token_embedding.weight"].grad.float()[used[:16]].numpy(),
        "token_rows_idx": used[:16].numpy(),
    }
    return res


def ddp_loss_worker(rank, world, port, feats, out_path):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    open_clip = import_reference()
    bl = feats["img"].shape[0] // world
    img = feats["img"][rank * bl:(rank + 1) * bl].clone().requires_grad_(True)
    txt = feats["txt"][rank * bl:(rank + 1) * bl].clone().requires_grad_(True)
    scale = feats["scale"].clone().requires_grad_(True)
    loss_fn = open_clip.ClipLoss(local_loss=True, gather_with_grad=True, rank=rank, world_size=world)
    loss = loss_fn(img, txt, scale)
    loss.backward()
    torch.save({"loss": loss.detach(), "d_img": img.grad, "d_txt": txt.grad, "d_scale": scale.grad},
               f"{out_path}.{rank}")
    dist.destroy_process_group()


def make_ddp_loss_golden():
    import torch.multiprocessing as mp
    g = torch.Generator().manual_seed(77)
    world, bl, E = 2, 12, 64
    img = torch.nn.functional.normalize(torch.randn(world * bl, E, generator=g), dim=-1)
    txt = torch.nn.functional.normalize(torch.randn(world * bl, E, generator=g), dim=-1)
    feats = {"img": img, "txt": txt, "scale": torch.tensor(14.2857)}
    tmp = tempfile.mkdtemp()
    out_path = os.path.join(tmp, "ddp")
    mp.spawn(ddp_loss_worker, args=(world, 29591, feats, out_path), nprocs=world, join=True)
    res = {"img": img.numpy(), "txt": txt.numpy(), "scale": feats["scale"].numpy(), "world": np.array(world)}
    for r in range(world):
        d = torch.load(f"{out_path}.{r}")
        res[f"loss_r{r}"] = d["loss"].numpy()
        res[f"d_img_r{r}"] = d["d_img"].numpy()
        res[f"d_txt_r{r}"] = d["d_txt"].numpy()
        res[f"d_scale_r{r}"] = d["d_scale"].numpy()
    np.savez_compressed(GOLD / "cliploss_world2_gloo.npz", **res)
    print("wrote cliploss_world2_gloo.npz", {k: float(res[k]) for k in ("loss_r0", "loss_r1")})


def make_schema_golden(open_clip):
    """state_dict keys / shapes and the dtype policy of precision='bf16' as the reference builds them
    (the drop-in contract for checkpoints and for the weight-decay split on parameter names)."""
    out = {}
    for name, cfg, image_size in (("tiny-cls", TINY_CONFIGS["tiny-cls"], 64), ("ViT-B-32-ctx16", CONFIG1, 192)):
        tmp = Path(tempfile.mkdtemp())
        (tmp / f"schema-{name}.json").write_text(json.dumps(cfg))
        open_clip.add_model_config(tmp)
        for precision in ("fp32", "bf16"):
            m = open_clip.create_model(f"schema-{name}", precision=precision, device="cpu",
                                       force_image_size=image_size, pos_embed="sin_cos_2d")
            out[f"{name}/{precision}"] = {
                "state_dict": {k: [list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()},
                "requires_grad": {k: bool(p.requires_grad) for k, p in m.named_parameters()},
                "buffers_non_persistent": [k for k, _ in m.named_buffers() if k not in m.state_dict()],
            }
    (GOLD / "reference_schema.json").write_text(json.dumps(out, indent=0))
    print("wrote reference_schema.json")


def make_host_ops_golden(open_clip):
    """Host-side pieces of the input/checkpoint stage (SURVEY 8f.4) run through the reference:
    PatchDropout (open_clip/transformer.py:53-90) with injected scores, and the position-table
    resamplers used when a checkpoint is loaded at another resolution / context length
    (open_clip/model.py:452-516)."""
    from types import SimpleNamespace
    from unittest import mock
    from open_clip.model import resize_pos_embed, resize_text_pos_embed
    from open_clip.transformer import PatchDropout
    g = torch.Generator().manual_seed(21)
    out = {}
    for tag, (b, n, d, prob) in {"pd_a": (3, 17, 8, 0.5), "pd_b": (2, 37, 4, 0.75), "pd_c": (4, 5, 6, 0.9)}.items():
        x = torch.randn(b, n, d, generator=g)
        scores = torch.randn(b, n - 1, generator=g)
        pd = PatchDropout(prob)
        pd.train()
        with mock.patch("torch.randn", return_value=scores):
            y = pd(x)
        out[f"{tag}_x"], out[f"{tag}_scores"], out[f"{tag}_y"] = x.numpy(), scores.numpy(), y.numpy()
        out[f"{tag}_prob"] = np.float64(prob)
    for tag, (og, ng, d) in {"pe_up": (6, 16, 32), "pe_down": (9, 6, 16)}.items():
        sd = {"visual.positional_embedding": torch.randn(1 + og * og, d, generator=g)}
        out[f"{tag}_old"] = sd["visual.positional_embedding"].numpy().copy()
        resize_pos_embed(sd, SimpleNamespace(visual=SimpleNamespace(grid_size=(ng, ng))))
        out[f"{tag}_new"] = sd["visual.positional_embedding"].numpy()
    for tag, (ol, nl, d) in {"te_up": (16, 32, 24), "te_down": (77, 16, 8)}.items():
        sd = {"positional_embedding": torch.randn(ol, d, generator=g)}
        out[f"{tag}_old"] = sd["positional_embedding"].numpy().copy()
        resize_text_pos_embed(sd, SimpleNamespace(positional_embedding=torch.zeros(nl, d)))
        out[f"{tag}_new"] = sd["positional_embedding"].numpy()
    np.savez_compressed(GOLD / "host_ops_ref.npz", **out)
    print("wrote host_ops_ref.npz")


def make_baseline_dim_goldens(open_clip):
    """fp32 and amp_bf16 reference runs at the BASELINE widths / head shapes / sequence lengths."""
    for i, (name, (cfg, image_size, pos_embed)) in enumerate(BASELINE_DIM_CASES.items()):
        for precision in ("fp32", "amp_bf16"):
            seed = 31 + i
            res = run_reference(open_clip, name, cfg, BASELINE_DIM_BATCH, image_size, pos_embed, seed, precision,
                                compact=True)
            meta = {"name": name, "batch": BASELINE_DIM_BATCH, "image_size": image_size, "pos_embed": pos_embed,
                    "seed": seed, "precision": precision, "cfg": cfg, "compact": True}
            meta["loss_dtype"] = res.pop("loss_dtype")
            np.savez_compressed(GOLD / f"{name}_{precision}.npz", meta=json.dumps(meta), **res)
            print(f"wrote {name}_{precision}.npz loss={float(res['loss']):.6f} ({meta['loss_dtype']})", flush=True)


def make_amp_goldens_small(open_clip):
    """amp_bf16 runs of the small cases (same-mode reference for the benchmarked precision)."""
    for (name, cfg, batch, image_size, pos_embed, seed) in CASES:
        res = run_reference(open_clip, name, cfg, batch, image_size, pos_embed, seed, "amp_bf16")
        meta = {"name": name, "batch": batch, "image_size": image_size, "pos_embed": pos_embed,
                "seed": seed, "precision": "amp_bf16", "cfg": cfg}
        meta["loss_dtype"] = res.pop("loss_dtype")
        np.savez_compressed(GOLD / f"{name}_amp_bf16.npz", meta=json.dumps(meta), **res)
        print(f"wrote {name}_amp_bf16.npz loss={float(res['loss']):.6f} ({meta['loss_dtype']})", flush=True)


def main():
    if "--baseline-dims-only" in sys.argv:
        torch.set_num_threads(os.cpu_count())
        oc = import_reference()
        make_amp_goldens_small(oc)
        make_baseline_dim_goldens(oc)
        return
    if "--schema-only" in sys.argv:
        GOLD.mkdir(parents=True, exist_ok=True)
        make_schema_golden(import_reference())
        return
    if "--host-ops-only" in sys.argv:
        GOLD.mkdir(parents=True, exist_ok=True)
        make_host_ops_golden(import_reference())
        return
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    GOLD.mkdir(parents=True, exist_ok=True)
    open_clip = import_reference()
    # pin the sin-cos restatement against the reference's own generator (open_clip/pos_embed.py:20)
    from open_clip.pos_embed import get_2d_sincos_pos_embed
    np.savez_compressed(GOLD / "sincos_ref.npz",
                        w128_g3=get_2d_sincos_pos_embed(128, 3, cls_token=True).astype(np.float32),
                        w768_g6=get_2d_sincos_pos_embed(768, 6, cls_token=True).astype(np.float32))
    for (name, cfg, batch, image_size, pos_embed, seed) in CASES:
        for precision in ("fp32", "bf16"):
            res = run_reference(open_clip, name, cfg, batch, image_size, pos_embed, seed, precision)
            meta = {"name": name, "batch": batch, "image_size": image_size, "pos_embed": pos_embed,
                    "seed": seed, "precision": precision, "cfg": cfg}
            loss_dtype = res.pop("loss_dtype")
            meta["loss_dtype"] = loss_dtype
            np.savez_compressed(GOLD / f"{name}_{precision}.npz", meta=json.dumps(meta), **res)
            print(f"wrote {name}_{precision}.npz loss={float(res['loss']):.6f} ({loss_dtype})")
    make_amp_goldens_small(open_clip)
    make_baseline_dim_goldens(open_clip)
    make_ddp_loss_golden()
    make_schema_golden(open_clip)
    make_host_ops_golden(open_clip)


if __name__ == "__main__":
    main()
