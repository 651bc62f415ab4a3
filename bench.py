#!/usr/bin/env python
"""Benchmark of the CLIPA training-step hot path (BASELINE.json metric: image-text pairs/sec at
ViT-L/14, global batch 32k, on 1/2/4/8 B200).

  python bench.py --gpus 1 --steps K --warmup W                  (single GPU)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...                           (CPU arm: the oracle port)

A "step" is one full optimizer step at the named global batch: H2D/preprocess (e2e only) ->
towers forward -> all-gather -> fused contrastive head -> backward -> gradient all-reduce ->
AdamW -> logit-scale clamp.  Global batch is FIXED as N grows ("strong" scaling): each rank
processes global/N pairs -- as one plain forward/backward when that fits 180 GB (4096 pairs of the
headline model: N = 8), otherwise in chunks with the reference's GradCache schedule (accum_freq
path); the chunk size (--micro-batch, default per workload) is the one at which every block can keep
its MLP activations, so backward skips the c_fc recompute GEMM.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# model, image px, pos-embed, global batch, algorithmic fwd+bwd GFLOP per pair (BASELINE.md section 3);
# micro = (largest per-GPU batch that runs as ONE plain forward/backward in 180 GB, chunk size when the per-GPU batch
# is larger than that and the GradCache schedule is needed anyway: small enough that the blocks keep their MLP
# activations, see Transformer._activation_policy)
WORKLOADS = {
    "vitl14_i81_t16_gb32k": dict(model="ViT-L-14-CL16", image=126, pos="sin_cos_2d", global_batch=32768,
                                 gflop_per_pair=159.35, baseline_config="configs[2]", micro=(4096, 2048)),
    "vitb16_i64_t16_gb16k": dict(model="ViT-B-16-CL16", image=128, pos="sin_cos_2d", global_batch=16384,
                                 gflop_per_pair=37.57, baseline_config="configs[1]", micro=(8192, 8192)),
    "vitl14_i256_t32_gb16k": dict(model="ViT-L-14-CL32", image=224, pos="learnable", global_batch=16384,
                                  gflop_per_pair=502.65, baseline_config="configs[3]", micro=(2048, 1024)),
    "vith14_i36_t8_gb64k": dict(model="ViT-H-14-CL8-SyntaxMask-GAP", image=84, pos="sin_cos_2d",
                                global_batch=65536, gflop_per_pair=155.84, baseline_config="configs[4]", micro=(8192, 4096)),
    # small plumbing case for smoke runs of this script
    "vitb32_i36_t16_gb256": dict(model="ViT-B-32-CL16", image=192, pos="sin_cos_2d", global_batch=256,
                                 gflop_per_pair=23.16, baseline_config="configs[0] shape, batch 256", micro=(256, 128)),
}
def pick_micro_batch(wl: dict, per_gpu_batch: int) -> int:
    """The whole per-GPU batch when it runs as one plain forward/backward, else the workload's GradCache chunk size."""
    plain, chunk = wl["micro"]
    return per_gpu_batch if per_gpu_batch <= plain else chunk


METRIC = "image-text pairs/sec at ViT-L/14, global batch 32k, 1/2/4/8 B200"


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d, "measured (MEASURED_PEAKS.json)"
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path (bounded sample of the same workload)
# ------------------------------------------------------------------------------------------------
def effective_cpus() -> int:
    """Host cores this process may actually use: min(affinity mask, cgroup CPU quota).  os.cpu_count()
    reports the machine's logical CPUs, which oversubscribes torch's thread pool inside a
    quota-limited container (measured: 128 threads on a throttled box ran 100x slower)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def cpu_step_fn(wl, batch):
    import torch
    from clipa_b200.open_clip import get_model_config
    from oracle import clip_oracle as O
    from oracle.weights import make_inputs, make_state_dict
    O.USE_FUSED = True   # same fused CPU primitives the reference calls (see oracle/clip_oracle.py)
    cfg = get_model_config(wl["model"])
    sd = make_state_dict(cfg, 0, image_size=wl["image"], pos_embed=wl["pos"])
    for v in sd.values():
        v.requires_grad_(True)
    images, text = make_inputs(cfg, batch, 1, image_size=wl["image"])

    def step():
        for v in sd.values():
            v.grad = None
        loss = O.train_step_loss(images, text, sd, cfg)
        loss.backward()
        return float(loss.detach())
    return step


def calibrated_cpu_step(wl, max_batch, target_s=5.0):
    """Pick the sample size (pairs per CPU step) so that one oracle step takes ~target_s seconds."""
    import torch
    cores = effective_cpus()
    torch.set_num_threads(cores)
    step1 = cpu_step_fn(wl, 1)
    step1()                       # first call pays allocator / thread-pool start-up
    t0 = time.perf_counter()
    step1()
    t1 = time.perf_counter() - t0
    batch = int(max(1, min(max_batch, target_s / max(t1, 1e-3))))
    return (step1 if batch == 1 else cpu_step_fn(wl, batch)), batch, cores


def cpu_baseline(wl, budget_s=20.0, batch=8):
    step, batch, cores = calibrated_cpu_step(wl, batch)
    step()  # warm-up
    t0 = time.perf_counter()
    n = 0
    while True:
        step(); n += 1
        if time.perf_counter() - t0 > budget_s or n >= 10:
            break
    dt = (time.perf_counter() - t0) / n
    return {"value": batch / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": f"oracle (oracle/clip_oracle.py) fwd+loss+bwd of {wl['model']} @{wl['image']}px, "
                      f"batch {batch}, {n} steps after 1 warm-up, fp32, torch CPU threads={cores}"}


DUMP_SAMPLE = 1 << 22     # parameter elements written by --dump-outputs (16 MB of float32)


def dump_outputs(out_dir: Path, loss, model) -> None:
    """What a caller of the timed step holds after its last step, as float32 .npy files: the loss it returned and the
    parameters it updated (logit_scale whole; the rest as a fixed, seeded sample of DUMP_SAMPLE elements of all
    parameters concatenated in named_parameters() order, in ascending position)."""
    import numpy as np
    import torch
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "loss.npy", np.asarray([float(loss)], dtype=np.float32))
    np.save(out_dir / "logit_scale.npy", model.logit_scale.detach().float().reshape(1).cpu().numpy())
    flat = [p.detach().reshape(-1) for _, p in model.named_parameters()]
    sizes = torch.tensor([t.numel() for t in flat])
    ends = torch.cumsum(sizes, 0)
    total = int(ends[-1])
    idx, _ = torch.sort(torch.randint(0, total, (min(DUMP_SAMPLE, total),), generator=torch.Generator().manual_seed(0)))
    lo, hi = torch.searchsorted(idx, ends - sizes).tolist(), torch.searchsorted(idx, ends).tolist()
    vals = torch.cat([t[(idx[a:b] - int(e - n)).to(t.device)].float().cpu()
                      for t, a, b, e, n in zip(flat, lo, hi, ends.tolist(), sizes.tolist())])
    np.save(out_dir / "params_sample.npy", vals.numpy())


def library_baseline_leg(wl, batch):
    """Bounded sample of the "library Blackwell path to beat" (SURVEY 8d): the unmodified reference
    (oracle/_ref) on torch's CUDA kernels, same box, right after our timed region.  Reported beside the
    headline, never part of it."""
    import gc
    import torch
    from baseline.ref_loader import available
    if not available():
        return {"unavailable": "oracle/_ref not installed (oracle/install_reference.sh)"}
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    try:
        from baseline.library_step import library_baseline
        r = library_baseline(wl, batch, steps=3, warmup=2)
        r["unit"] = "pairs/s"
        r["value"] = r.pop("pairs_per_s")
        return r
    except Exception as e:  # noqa: a failure of the comparison arm must not lose the measurement
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}


def run_reference_arm(args, wl, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    step, batch, cores = calibrated_cpu_step(wl, args.cpu_batch)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = batch / dt
    sample = (f"each step = oracle port of the reference path, {wl['model']} @{wl['image']}px, batch {batch} "
              f"(bounded sample of the {wl['global_batch']}-pair step), fp32, torch CPU threads={cores}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": name, "model": wl["model"], "global_batch": wl["global_batch"], "cpu_batch": batch},
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="vitl14_i81_t16_gb32k", choices=list(WORKLOADS))
    ap.add_argument("--global-batch", type=int, default=None)
    ap.add_argument("--micro-batch", type=int, default=0,
                    help="pairs per forward/backward chunk (0 = auto from the workload's `micro` pair: the whole per-GPU "
                         "batch when it fits one plain step, else the GradCache chunk size at which the blocks keep "
                         "their MLP activations and backward skips the c_fc recompute GEMM)")
    ap.add_argument("--keep-mlp", default="auto", help="blocks that keep their MLP activations (auto | integer)")
    ap.add_argument("--precision", default="amp_bf16", choices=["amp_bf16", "bf16"])
    ap.add_argument("--cpu-batch", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true",
                    help="skip the bounded run of the unmodified reference on torch's CUDA kernels (N=1 only)")
    ap.add_argument("--library-batch", type=int, default=1024)
    ap.add_argument("--save-ln", default="auto", choices=["auto", "on", "off"],
                    help="keep LayerNorm outputs for backward (auto: when HBM allows)")
    ap.add_argument("--op-table", default=None, help="write the per-kernel CUDA-event table (JSON) to this path")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the last step's loss and updated parameters (a fixed sample) "
                         "to DIR/*.npy, to compare two builds output for output")
    args = ap.parse_args()
    name = args.workload
    wl = dict(WORKLOADS[name])
    if args.global_batch:
        wl["global_batch"] = args.global_batch
    if args.impl == "reference":
        run_reference_arm(args, wl, name)
        return

    import torch
    import torch.distributed as dist
    from clipa_b200 import _lib, open_clip, ops
    from clipa_b200.training import TrainStep

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    gb = wl["global_batch"]
    assert gb % world == 0
    bl = gb // world
    torch.manual_seed(0)
    model, _, _ = open_clip.create_model_and_transforms(wl["model"], precision=args.precision, device=dev,
                                                        force_image_size=wl["image"], pos_embed=wl["pos"],
                                                        output_dict=True)
    if world > 1:  # identical replicas (DDP's initial broadcast, training/main.py:299)
        for p in model.parameters():
            dist.broadcast(p.data, 0)
    from clipa_b200.open_clip.transformer import Transformer as _T
    _T.save_ln_outputs = {"auto": "auto", "on": True, "off": False}[args.save_ln]
    _T.keep_mlp_blocks = "auto" if args.keep_mlp == "auto" else int(args.keep_mlp)
    if args.micro_batch <= 0:
        args.micro_batch = pick_micro_batch(wl, bl)
    model.train()
    trainer = TrainStep(model, rank=rank, world_size=world, micro_batch=args.micro_batch,
                        overlap_grad_allreduce=os.environ.get("CLIPA_OVERLAP", "0") == "1")
    ctx = model.context_length
    vocab = model.vocab_size
    g = torch.Generator().manual_seed(1 + rank)
    # host buffers in pinned memory: uint8 images (--to-float-on-device recipe) and int64 token ids
    h_images = torch.randint(0, 256, (bl, 3, wl["image"], wl["image"]), generator=g, dtype=torch.uint8).pin_memory()
    h_text = torch.randint(1, vocab - 1, (bl, ctx), generator=g, dtype=torch.int64)
    h_text[:, -1] = vocab - 1
    h_text = h_text.pin_memory()
    d_images = trainer.preprocess(h_images)      # resident, already normalised bf16
    d_text = h_text.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        n0 = _lib.launch_count()
        if profile:
            ops.PROFILER = ops.GemmProfiler()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        barrier()
        prof, ops.PROFILER = ops.PROFILER, None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        clocks = sampler.stop() if rank == 0 else None
        return ms.item() / steps, _lib.launch_count() - n0, clocks, prof, last

    # ---- device-resident throughput (`value`): uninstrumented region ----
    ms_step, launches, clocks, _, last_loss = timed(lambda: trainer.step(d_images, d_text), args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), last_loss, model)
    value = gb / (ms_step * 1e-3)
    # ---- second pass with the per-launch CUDA-event profiler on: roofline of the GEMM kernels + op table ----
    prof_steps = max(1, args.steps // 2)
    ms_prof, _, _, prof, _ = timed(lambda: trainer.step(d_images, d_text), prof_steps, 0, profile=True)
    gemm_tflops, gemm_ms, gemm_calls = prof.summary()
    rows = prof.table()
    attn_bwd_flops = sum(r["tflops"] * r["ms"] * 1e9 for r in rows if r["key"][0] == "attn_bwd")   # FLOP over the pass
    if args.op_table and rank == 0:
        Path(args.op_table).parent.mkdir(parents=True, exist_ok=True)
        Path(args.op_table).write_text(json.dumps({"steps": prof_steps, "ms_per_step": ms_prof,
                                                   "ms_per_step_uninstrumented": ms_step, "rows": rows}, indent=1))

    # ---- end-to-end through the public step with HOST buffers (`e2e`) ----
    e2e = None
    if not args.no_e2e:
        def e2e_step():
            loss = trainer.step(h_images, h_text)       # pinned host -> device inside the step
            return loss.item()                           # device -> host read of the result
        ms_e2e, _, _, _, _ = timed(e2e_step, max(2, args.steps // 2), 1)
        e2e = {"value": gb / (ms_e2e * 1e-3), "unit": "pairs/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": (h_images.numel() + h_text.numel() * 8) * world,
               "d2h_bytes_per_step": 4 * world,
               "steps": max(2, args.steps // 2), "warmup": 1,
               "note": "h2d = uint8 images + int64 token ids from pinned memory, all ranks; d2h = loss scalar"}

    if rank == 0:
        pk, pk_src = peaks()
        peak = pk["bf16_tflops_sustained"]
        # dram__bytes_read.sum + dram__bytes_write.sum of the largest-share GEMM launch, from the committed
        # ncu --set full capture (profiles/ncu_traffic.json names the capture); absent -> null
        try:
            traffic = json.loads((Path(__file__).resolve().parent / "profiles" / "ncu_traffic.json").read_text())
        except (OSError, ValueError):
            traffic = {}
        per_gpu_pairs = value / world
        # algorithmic GEMM work of one step on this GPU: BASELINE.md's fwd+bwd FLOP per pair (no recompute, one
        # forward per pair) minus the attention-core share (3.5/2.5 x the executed attention-backward FLOP)
        alg_total = wl["gflop_per_pair"] * 1e9 * bl
        alg_gemm = alg_total - 1.4 * attn_bwd_flops / prof_steps
        gemm_s_per_step = gemm_ms / prof_steps * 1e-3
        frac_alg = alg_gemm / gemm_s_per_step / 1e12 / peak if gemm_s_per_step > 0 else None
        out = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": name, "baseline_config": wl["baseline_config"], "model": wl["model"],
                       "image_px": wl["image"], "image_tokens_incl_cls": model.visual.positional_embedding.shape[0],
                       "text_tokens": ctx, "global_batch": gb, "per_gpu_batch": bl,
                       "micro_batch": min(bl, args.micro_batch),
                       "schedule": "plain fwd/bwd" if bl <= args.micro_batch else "GradCache (N chunks: N-1 no-grad forwards + N fwd/bwd; last chunk keeps its graph)",
                       "parallelism": f"dp{world}", "precision": args.precision,
                       "optimizer": "AdamW (clipa_adamw_step: fused update + bf16 shadow + grad clear) inside the timed step", "l2": "inputs_exceed_L2",
                       "loss_last": float(last_loss),
                       "peak_hbm_gb": round(torch.cuda.max_memory_allocated(dev) / 2**30, 1),
                       "save_ln_outputs": str(type(model.visual.transformer).save_ln_outputs),
                       "activation_policy_vision(save_ln,drop_o,keep_mlp_blocks)": list(getattr(model.visual.transformer, "last_policy", ())),
                       "activation_policy_text(save_ln,drop_o,keep_mlp_blocks)": list(getattr(model.transformer, "last_policy", ())),

                       "algorithmic_gflop_per_pair": wl["gflop_per_pair"],
                       "model_flops_utilization": per_gpu_pairs * wl["gflop_per_pair"] / (peak * 1e3)},
            "clocks": clocks, "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "gemm_tc2_kernel / gemm_tc_kernel (tcgen05, all epilogues/majors)",
                         "achieved": gemm_tflops, "peak": peak, "unit": "TFLOP/s", "frac": gemm_tflops / peak,
                         "frac_executed": gemm_tflops / peak, "frac_algorithmic": frac_alg,
                         "note": "frac/frac_executed count every GEMM launch (incl. the c_fc recompute in backward and "
                                 "GradCache's extra forwards); frac_algorithmic counts only BASELINE.md's FLOP per pair",
                         "traffic": traffic.get("dram_bytes_per_launch"), "traffic_of": traffic.get("of"),
                         "peak_source": pk_src + ", sustained figure (kernel timed inside a long step)",
                         "gemm_launches_timed": gemm_calls, "gemm_ms_per_step": gemm_ms / prof_steps,
                         "gemm_share_of_step": gemm_ms / prof_steps / ms_prof,
                         "measured_in": f"second pass of {prof_steps} step(s) with per-launch CUDA events "
                                        f"({ms_prof:.1f} ms/step vs {ms_step:.1f} uninstrumented)"},
        }
        if e2e:
            out["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(wl, batch=args.cpu_batch)
        if world == 1 and not args.no_library_baseline:
            # release OUR model, optimizer state and activations first: the comparison arm gets the whole GPU
            trainer.model = None
            del trainer, model, d_images, d_text
            out["library_baseline"] = library_baseline_leg(wl, args.library_batch)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
