"""Generates tests/golden/reference_caller.json on a CUDA device: runs the UNMODIFIED reference's own caller code over
clipa_b200.open_clip aliased as `open_clip` (INTEGRATION.md section 1) on the seeded models, batches and optimizer
settings of tests/test_reference_caller_gpu.py, and stores what that test compares against:
  train_one_epoch/<accum_freq>  the Contrastive_loss training/train.py `train_one_epoch` logs at every optimizer step
                                over 3 epochs of 6 batches (accum_freq 1 and 2), and the final logit_scale
  zero_shot                     top-1 / top-5 accuracy of training/zero_shot.py `run`
It also prints what TrainStep and clipa_b200.zero_shot give on the same inputs.

The reference is imported from oracle/_ref (oracle/install_reference.sh).
Usage:  python oracle/make_caller_golden.py [out.json]      (default tests/golden/reference_caller.json)
"""
from __future__ import annotations

import contextlib
import importlib
import importlib.machinery
import json
import logging
import subprocess
import sys
from pathlib import Path
from unittest.mock import MagicMock

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from tests import test_reference_caller_gpu as T  # noqa: E402  (the recipe the golden is compared under)


@contextlib.contextmanager
def reference_over_alias():
    """Imports the reference's `training` package with `open_clip` resolving to clipa_b200.open_clip."""
    from baseline import ref_loader
    root = ref_loader.reference_root()
    if root is None:
        raise SystemExit(f"reference not installed in {ref_loader.REF_DIR}: run oracle/install_reference.sh")
    import clipa_b200.open_clip as ours
    # stubs for the tokenizer / data-loader dependencies that are not installed (see baseline/ref_loader.py)
    for n in ref_loader._STUBS:
        if n not in sys.modules:
            try:
                __import__(n)
            except Exception:
                m = MagicMock()
                m.__spec__ = importlib.machinery.ModuleSpec(n, None)
                m.__path__ = []
                sys.modules[n] = m
    sys.modules["open_clip"] = ours
    for sub in ("factory", "model", "loss", "transformer", "pos_embed", "model_configs"):
        sys.modules[f"open_clip.{sub}"] = importlib.import_module(f"clipa_b200.open_clip.{sub}")
    sys.path.insert(0, str(root))
    try:
        train = importlib.import_module("training.train")
        zero_shot = importlib.import_module("training.zero_shot")
        data = importlib.import_module("training.data")
        assert train.CLIP is ours.CLIP                      # train.py:28 imported OUR classes
        yield train, zero_shot, data
    finally:
        sys.path.remove(str(root))


class _Capture(logging.Handler):
    def __init__(self):
        super().__init__(logging.INFO)
        self.messages = []

    def emit(self, record):
        self.messages.append(record.getMessage())


def reference_train_one_epoch(ref, dev, accum_freq):
    train, _, data = ref
    from clipa_b200 import open_clip
    args = T._args(dev, accum_freq, T.BS)
    model = T._build_model(dev, args)
    optimizer = T._build_optimizer(model, args)
    loss = open_clip.create_loss(args)
    batches = T._batches(T.N_BATCHES, T.BS, model.vocab_size)
    loaders = {"train": data.DataInfo(dataloader=T._Loader(batches, T.BS))}
    cap = _Capture()
    root = logging.getLogger()
    old_level = root.level
    root.addHandler(cap)
    root.setLevel(logging.INFO)
    try:
        for epoch in range(T.EPOCHS):
            train.train_one_epoch(model, loaders, loss, epoch, optimizer, None, None, None, args)
    finally:
        root.removeHandler(cap)
        root.setLevel(old_level)
    torch.cuda.synchronize()
    logged = [float(m.split("Contrastive_loss: ")[1].split()[0]) for m in cap.messages if "Contrastive_loss" in m]
    return {"logged": logged, "logit_scale": model.logit_scale.item()}


def reference_zero_shot(ref, dev):
    _, zero_shot, _ = ref
    from clipa_b200 import zero_shot as zs
    args = T._args(dev, 1, 8)
    model = T._build_model(dev, args)
    model.eval()
    ids, loader = T._zero_shot_inputs(model)
    classifier = zs.zero_shot_classifier(model, class_token_ids=ids)
    top1, top5 = zero_shot.run(model, classifier.float(), loader, args)
    return {"top1": float(top1), "top5": float(top5)}


def device_description(dev) -> str:
    """GPU name and power limit: the golden losses carry bf16 and fp32-atomic noise of the device they ran on."""
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev.index)],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        limit = ""
    return f"{torch.cuda.get_device_name(dev)}, power limit {limit or 'unknown'}"


def main():
    out = Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "tests" / "golden" / "reference_caller.json"
    dev = torch.device("cuda:0")
    with reference_over_alias() as ref:
        gold = {"train_one_epoch": {str(a): reference_train_one_epoch(ref, dev, a) for a in (1, 2)},
                "zero_shot": reference_zero_shot(ref, dev),
                "device": device_description(dev)}
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(gold, indent=1) + "\n")
    print(f"wrote {out}")
    for a in (1, 2):
        model, _, ours = T.train_trajectory(dev, a)
        ref_losses = gold["train_one_epoch"][str(a)]["logged"]
        rel = [abs(x - y) / abs(y) for x, y in zip(ours, ref_losses)]
        print(f"accum_freq {a}: reference {ref_losses}\n  TrainStep {ours}\n  max rel diff {max(rel):.3e}; "
              f"logit_scale {model.logit_scale.item():.6f} vs {gold['train_one_epoch'][str(a)]['logit_scale']:.6f}")
    _, _, top1, top5 = T.zero_shot_accuracy(dev)
    print(f"zero-shot: reference {gold['zero_shot']}, ours top1 {top1} top5 {top5}")


if __name__ == "__main__":
    main()
