#!/usr/bin/env python
"""Benchmark of the CLIP contrastive training hot path (fwd + bwd), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): image-text pairs/s (fwd+bwd) at global batch 32768.  A "step" is one
`loss = clip(text, images, return_loss=True); loss.backward()` on one batch of synthetic data
(text = randint, images = randn, reference default init).

Default workload = cfg3 of BASELINE.json, the configuration the metric is quoted on: ViT-B/16 image
tower (dim 768, 12 layers, 12 heads, 224 px / patch 16, reference-default visual_patch_dropout 0.5)
+ 12-layer text tower (dim 512, 77 tokens), dim_latent 512, plain InfoNCE, 4096 pairs per GPU
(global batch 4096*N: 32768 at N = 8, weak scaling, negatives all-gathered across ranks), encoder
micro-batch 768 (GradCache-style step, engine.ChunkedClipLossFn: 4096 pairs of ViT-B/16 activations are
~260 GB; the chunks that fit the 180 GB of HBM keep their activations, the rest is re-encoded in backward;
the reference's own answer is activation checkpointing).

One JSON line on rank 0:
  value        pairs/s with the batch already on the device
  e2e          the same step through the public CLIP.forward with the batch copied from pinned
               host memory inside the timed region (double buffered, side stream) + loss read-back
  roofline     the dominant kernel family (tcgen05 GEMM) measured live with CUDA events around every
               C-ABI call in one instrumented step, plus `attention` and `logits` sub-objects (the
               kernels the north star names): tensor-pipe fraction AND achieved HBM GB/s
  cpu_baseline the UNMODIFIED reference (oracle/_ref, pip-installed from /root/reference) on the
               host cores, bounded sample of the same model; `gpu_eager_baseline`: the unmodified
               reference module on this B200 in eager PyTorch (fp32 and bf16 autocast)
  other_workloads  short measurements of cfg2 (README model, 1024/GPU), cfg4 (FILIP, 256/GPU) and
               cfg5 (DCL + extra projections, 8192/GPU) on the same N GPUs
  multirank_parity (N > 1) per-rank loss / grad-norm / d temperature of a tiny sharded step against
               the oracle's restatement of the reference's per-rank contract (distributed.py:41-56)
`--impl reference` times the reference's own CPU implementation of the same model on the host.
`--dump-outputs DIR` writes what the last device-resident timed step returned to its caller: the loss
and every parameter gradient, as DIR/loss.npy and DIR/grad.<parameter name>.npy (float32; a fixed,
seeded sample of each large gradient, at most 64 MB in all).  Same arguments give the same inputs, so
the dumps of two builds can be compared array by array.
"""
from __future__ import annotations

import argparse
import atexit
import json
import math
import os
import subprocess
import sys
import threading
import time
import zlib
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

README_CFG = dict(dim_text=512, dim_image=512, dim_latent=512, num_text_tokens=10000,
                  text_enc_depth=6, text_seq_len=256, text_heads=8, visual_enc_depth=6,
                  visual_image_size=256, visual_patch_size=32, visual_heads=8)
# cfg3 of BASELINE.json: ViT-B/16 image tower + 12-layer text tower (CLIP tokenizer vocabulary)
VITB16_CFG = dict(dim_text=512, dim_image=768, dim_latent=512, num_text_tokens=49408,
                  text_enc_depth=12, text_seq_len=77, text_heads=8, visual_enc_depth=12,
                  visual_image_size=224, visual_patch_size=16, visual_heads=12)
METRIC = "image-text pairs/sec (fwd+bwd)"
WORKLOADS = {
    "cfg2": (README_CFG, "cfg2: README CLIP (dim 512, text 6L seq 256, ViT 6L 256px/32, 8 heads, "
                         "visual_patch_dropout {pd} (reference default 0.5), {loss}), {b} pairs/GPU"),
    "cfg3": (VITB16_CFG, "cfg3: ViT-B/16 (dim 768, 12L, 12 heads, 224px/16) + text 12L dim 512 seq 77, "
                         "dim_latent 512, visual_patch_dropout {pd}, {loss}, {b} pairs/GPU"),
}
LOSS_KW = {"nce": {}, "dcl_extra": dict(decoupled_contrastive_learning=True, extra_latent_projection=True),
           "filip": dict(use_all_token_embeds=True)}
LOSS_TXT = {"nce": "plain InfoNCE", "dcl_extra": "DCL + extra latent projection",
            "filip": "FILIP (use_all_token_embeds)"}
DEFAULTS = {"cfg3": dict(batch=4096, microbatch=768), "cfg2": dict(batch=1024, microbatch=0)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="pairs per GPU (default: 4096 cfg3, 1024 cfg2)")
    ap.add_argument("--microbatch", type=int, default=None,
                    help="encoder micro-batch of the GradCache-style step (default: 768 cfg3, off cfg2)")
    ap.add_argument("--retain", default="auto",
                    help="micro-batched step: chunks whose activations stay resident in HBM between the "
                         "forward and the backward sweep ('auto' = as many as fit, 0 = pure two-pass step)")
    ap.add_argument("--tune", default="", help="A/B switches 'knob=value,...' passed to xclip_tune_set")
    ap.add_argument("--patch-dropout", type=float, default=0.5)
    ap.add_argument("--loss", default="nce", choices=sorted(LOSS_KW))
    ap.add_argument("--grad-sync", action="store_true",
                    help="N>1: also all-reduce the weight gradients inside the timed step "
                         "(x_clip_b200.distributed.GradSync, buckets overlapped with backward); the "
                         "reference leaves this to the user's DDP wrapper")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg2 / cfg4 / cfg5 side measurements")
    ap.add_argument("--no-parity", action="store_true", help="skip the N>1 per-rank parity check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and the parameter gradients of the last timed step to DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs dumps the GPU step (--impl ours)")
    a.retain = a.retain if a.retain == "auto" else int(a.retain)
    d = DEFAULTS[a.workload]
    if a.batch is None:
        a.batch = d["batch"] if a.loss == "nce" else {"filip": 256, "dcl_extra": 8192}[a.loss]
    if a.microbatch is None:
        a.microbatch = d["microbatch"] if a.loss == "nce" else {"filip": 0, "dcl_extra": 1024}[a.loss]
    return a


def workload_text(args, batch=None, plan=None):
    cfg, txt = WORKLOADS[args.workload]
    s = txt.format(b=batch or args.batch, pd=args.patch_dropout, loss=LOSS_TXT[args.loss])
    if args.microbatch:
        s += f", encoder micro-batch {args.microbatch} (GradCache-style step"
        if plan:
            s += (f": activations of {plan['retained']} of {plan['chunks']} chunks stay in HBM, the other "
                  f"{plan['chunks'] - plan['retained']} are re-encoded in backward = +{plan['chunks'] - plan['retained']}"
                  f"/{plan['chunks']} encoder forward")
        s += ")"
    return s


# --------------------------------------------------------------------------- CPU arm (reference)

def _reference_module(model_cfg, loss_kw, patch_dropout, device="cpu"):
    """The UNMODIFIED reference CLIP (oracle/_ref) with its own default initialisation; falls back
    to None when oracle/_ref was never built (then the oracle port is timed instead)."""
    try:
        from oracle import build_ref
        x_clip = build_ref.import_reference()
    except Exception:
        return None
    import torch
    torch.manual_seed(0)
    clip = x_clip.CLIP(**model_cfg, **loss_kw, visual_patch_dropout=patch_dropout,
                       use_mlm=False, use_visual_ssl=False).to(device)
    clip.train()
    return clip


def cpu_reference_rate(model_cfg, loss_kw, patch_dropout, batch, steps, warmup, budget_s):
    """pairs/s of the reference's own CLIP.forward(return_loss=True) + backward, fp32, on the host
    cores; `batch` pairs per step (a bounded sample of the workload).  -> dict"""
    import torch
    cores = min(os.cpu_count() or 1, 32)   # beyond ~32 threads intra-op scaling of these shapes degrades
    torch.set_num_threads(cores)
    clip = _reference_module(model_cfg, loss_kw, patch_dropout)
    kind = "reference"
    if clip is None:                        # oracle port (same arithmetic, functional restatement)
        from oracle import clip_oracle as O
        kind = "port"
        cfg = O.ClipConfig(**model_cfg, **loss_kw)
        state = O.protocol_state_dict(cfg, 1234)
        params = {k: v.clone().requires_grad_(True) for k, v in state.items()}
        n_patch = (cfg.visual_image_size // cfg.visual_patch_size) ** 2
    g = torch.Generator().manual_seed(7)
    times, t_start = [], time.time()
    for i in range(warmup + steps):
        text = torch.randint(0, model_cfg["num_text_tokens"], (batch, model_cfg["text_seq_len"]), generator=g)
        image = torch.randn(batch, 3, model_cfg["visual_image_size"], model_cfg["visual_image_size"], generator=g)
        t0 = time.perf_counter()
        if kind == "reference":
            loss = clip(text, image, return_loss=True)
            loss.backward()
            clip.zero_grad(set_to_none=True)
        else:
            keep = None
            if patch_dropout > 0:
                keep = torch.randn(batch, n_patch).topk(max(1, int(n_patch * (1 - patch_dropout))), dim=-1).indices
            loss = O.clip_forward(params, text, image, cfg, keep=keep)
            loss.backward()
            for v in params.values():
                v.grad = None
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        if time.time() - t_start > budget_s and len(times) >= 1:
            break
    ms = 1e3 * sum(times) / len(times)
    return dict(value=batch / (ms / 1e3), ms=ms, cores=cores, steps=len(times), kind=kind, batch=batch)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model_cfg, _ = WORKLOADS[args.workload]
    batch = 8
    r = cpu_reference_rate(model_cfg, LOSS_KW[args.loss], args.patch_dropout, batch, args.steps,
                           min(args.warmup, 2), budget_s=150.0)
    what = ("the unmodified reference (oracle/_ref, x_clip.CLIP.forward + backward)" if r["kind"] == "reference"
            else "the oracle port of the reference")
    sample = (f"{r['steps']} steps of {batch} pairs (fwd+bwd, fp32, same model as the GPU arm, "
              f"patch dropout {args.patch_dropout}), {r['ms']:.0f} ms/step")
    line = {
        "impl": "reference", "metric": METRIC, "value": round(r["value"], 3), "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": min(args.warmup, 2),
        "ms_per_step": round(r["ms"], 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args), "sample_batch": batch,
                   "note": f"CPU arm: {what}, all host threads (capped at 32)"},
        "cpu_baseline": {"value": round(r["value"], 3), "unit": "pairs/s", "cores": r["cores"],
                         "kind": r["kind"], "sample": sample},
        "e2e": {"value": round(r["value"], 3), "unit": "pairs/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- clocks

class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            atexit.register(self.proc.kill)     # never outlive the benchmark, even when it fails
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        busy = [x for x in sm if x > 0.5 * (mx[0] if mx else 1)] or sm
        return {"sm_mhz": busy[len(busy) // 2] if busy else None,
                "sm_max_mhz": mx[0] if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------- GPU arm helpers

class Runner:
    """One model + synthetic data on this rank; `timed(steps)` -> ms for `steps` device-resident steps
    (CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks)."""

    def __init__(self, model_cfg, loss, batch, microbatch, patch_dropout, dev, rank, world, grad_sync=False,
                 host_buffers=0, retain="auto"):
        import torch
        import x_clip_b200
        self.torch, self.dev, self.rank, self.world, self.B = torch, dev, rank, world, batch
        self.cfg = model_cfg
        torch.manual_seed(0)
        self.clip = x_clip_b200.CLIP(**model_cfg, **LOSS_KW[loss], visual_patch_dropout=patch_dropout,
                                     microbatch=microbatch or None, microbatch_retain=retain).to(dev)
        self.clip.train()
        self.params = list(self.clip.parameters())
        self.host = []
        S, V, I = model_cfg["text_seq_len"], model_cfg["num_text_tokens"], model_cfg["visual_image_size"]
        if host_buffers:
            g = torch.Generator().manual_seed(1 + rank)
            t0 = torch.randint(0, V, (batch, S), generator=g).pin_memory()
            im0 = torch.empty(batch, 3, I, I).pin_memory()
            torch.randn(im0.shape, generator=g, out=im0)
            self.host.append((t0, im0))
            for _ in range(host_buffers - 1):          # further buffers: the same samples, batch order flipped
                t1 = torch.empty_like(t0).pin_memory(); t1.copy_(t0.flip(0))
                im1 = torch.empty_like(im0).pin_memory(); im1.copy_(im0.flip(0))
                self.host.append((t1, im1))
            self.text, self.image = self.host[0][0].to(dev), self.host[0][1].to(dev)
        else:
            gd = torch.Generator(device=dev).manual_seed(1 + rank)
            self.text = torch.randint(0, V, (batch, S), generator=gd, device=dev)
            self.image = torch.randn(batch, 3, I, I, generator=gd, device=dev)
        self.grad_sync = None
        if grad_sync and world > 1:
            from x_clip_b200.distributed import GradSync
            self.grad_sync = GradSync(self.clip)

    def step(self, text=None, image=None):
        for p in self.params:
            p.grad = None
        loss = self.clip(self.text if text is None else text, self.image if image is None else image,
                         return_loss=True)
        loss.backward()
        if self.grad_sync is not None:
            self.grad_sync.finish()
        return loss

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms: float) -> float:
        if self.world == 1:
            return ms
        import torch.distributed as dist
        t = self.torch.tensor([ms], device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def timed(self, steps, warmup):
        torch = self.torch
        for _ in range(max(warmup, 1)):
            self.step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(steps):
            loss = self.step()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)), loss.item()

    def close(self):
        if self.grad_sync is not None:
            self.grad_sync.remove()
        self.clip = self.params = self.text = self.image = self.host = None
        self.torch.cuda.empty_cache()


DUMP_VALUES = 8 * 2**20     # sampled gradient values, float32: 32 MB, plus <= 4096 per tensor (64 MB cap)


def step_outputs(loss, clip):
    """-> {name: float32 numpy array} of what one step hands its caller: the loss and each parameter's
    gradient.  A gradient larger than its share of DUMP_VALUES is sampled at sorted positions drawn
    without replacement from a generator seeded by the parameter name, the same positions in every run."""
    import numpy as np
    import torch
    grads = [(n, p.grad) for n, p in clip.named_parameters() if p.grad is not None]
    frac = min(1.0, DUMP_VALUES / sum(g.numel() for _, g in grads))
    out = {"loss": np.asarray(loss.item(), dtype=np.float32)}
    for name, g in grads:
        flat = g.detach().float().reshape(-1)
        k = min(flat.numel(), max(4096, math.ceil(flat.numel() * frac)))
        if k < flat.numel():
            gen = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            idx = torch.randperm(flat.numel(), generator=gen)[:k].sort().values
            flat = flat[idx.to(flat.device)]
        out[f"grad.{name}"] = flat.cpu().numpy()
    assert sum(a.nbytes for a in out.values()) <= 64 * 2**20
    return out


def multirank_parity(dev, rank, world):
    """Tiny sharded step on all `world` ranks vs the oracle's restatement of the reference's per-rank
    contract (global loss on every rank; latent gradients of the LOCAL shard; full d temperature),
    and, at world = 2, vs the committed 2-rank run of the reference itself (tests/golden)."""
    import torch
    import torch.distributed as dist
    import x_clip_b200
    from oracle import clip_oracle as O      # checker only (never timed, never on the product path)
    gold_file = ROOT / "tests" / "golden" / "sharded_plain.json"
    gold = json.loads(gold_file.read_text())
    cfg = O.ClipConfig(**gold["cfg"])
    per = gold["per_rank"]
    state = O.protocol_state_dict(cfg, gold["weight_seed"])
    text, image = O.protocol_inputs(cfg, world * per, gold["input_seed"], gold["pad_fraction"])
    texts, images = list(text.chunk(world)), list(image.chunk(world))
    clip = x_clip_b200.CLIP(**gold["cfg"], visual_patch_dropout=0.).to(dev)
    clip.load_state_dict(state)
    clip.train()
    loss = clip(texts[rank].to(dev), images[rank].to(dev), return_loss=True)
    loss.backward()
    gn = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in clip.parameters() if p.grad is not None)).item()
    dt = clip.temperature.grad.item()
    p = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    o_loss = O.clip_forward_sharded(p, texts, images, cfg, rank)
    o_loss.backward()
    o_gn = torch.sqrt(sum((v.grad.double() ** 2).sum() for v in p.values() if v.grad is not None)).item()
    o_dt = p["temperature"].grad.item()
    rec = dict(rank=rank, loss=loss.item(), oracle_loss=o_loss.item(), grad_norm=gn, oracle_grad_norm=o_gn,
               dtemp=dt, oracle_dtemp=o_dt)
    if world == 2:
        rec["reference_loss"] = gold["ranks"][rank]["loss"]
        rec["reference_grad_norm"] = gold["ranks"][rank]["grad_norm"]
    recs = [None] * world
    dist.all_gather_object(recs, rec)
    loss_rel = max(abs(r["loss"] - r["oracle_loss"]) / abs(r["oracle_loss"]) for r in recs)
    gn_rel = max(abs(r["grad_norm"] - r["oracle_grad_norm"]) / r["oracle_grad_norm"] for r in recs)
    dt_abs = max(abs(r["dtemp"] - r["oracle_dtemp"]) for r in recs)
    out = dict(world=world, pairs_per_rank=per, max_loss_rel_err=loss_rel, max_grad_norm_rel_err=gn_rel,
               max_dtemp_abs_err=dt_abs, same_loss_on_all_ranks=max(r["loss"] for r in recs) - min(r["loss"] for r in recs) < 1e-6,
               checked_against="oracle restatement of the per-rank contract (x_clip/distributed.py:41-56)")
    if world == 2:
        out["max_loss_rel_err_vs_reference_2rank_run"] = max(
            abs(r["loss"] - r["reference_loss"]) / abs(r["reference_loss"]) for r in recs)
        out["max_grad_norm_rel_err_vs_reference_2rank_run"] = max(
            abs(r["grad_norm"] - r["reference_grad_norm"]) / r["reference_grad_norm"] for r in recs)
    out["ok"] = bool(loss_rel <= 1e-3 and gn_rel <= 2e-2 and out["same_loss_on_all_ranks"])
    del clip
    torch.cuda.empty_cache()
    return out


def gpu_eager_baseline(model_cfg, loss_kw, patch_dropout, dev, batch=256):
    """The UNMODIFIED reference module (oracle/_ref) on this GPU, eager PyTorch, fwd+bwd."""
    import torch
    clip = _reference_module(model_cfg, loss_kw, patch_dropout, device=dev)
    if clip is None:
        return {"unavailable": "oracle/_ref not built"}
    g = torch.Generator(device=dev).manual_seed(3)
    text = torch.randint(0, model_cfg["num_text_tokens"], (batch, model_cfg["text_seq_len"]), generator=g, device=dev)
    image = torch.randn(batch, 3, model_cfg["visual_image_size"], model_cfg["visual_image_size"], generator=g, device=dev)
    out = {"batch": batch, "what": "unmodified reference x_clip.CLIP (oracle/_ref), eager PyTorch on this B200, "
                                   "fwd+bwd, same model / patch dropout as the headline"}

    def run(autocast):
        def one():
            clip.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                loss = clip(text, image, return_loss=True)
            loss.backward()
        for _ in range(2):
            one()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            one()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 3
    try:
        ms = run(False)
        out["fp32_pairs_per_s"] = round(batch / (ms / 1e3), 1)
        out["fp32_ms_per_step"] = round(ms, 2)
        ms = run(True)
        out["bf16_autocast_pairs_per_s"] = round(batch / (ms / 1e3), 1)
        out["bf16_autocast_ms_per_step"] = round(ms, 2)
    except Exception as e:            # e.g. out of memory: report, do not kill the bench
        out["error"] = f"{type(e).__name__}: {str(e)[:200]}"
    del clip
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------- GPU arm

def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - x_clip_b200 has no CPU path "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    t_start = time.time()

    def note(msg):
        if os.environ.get("XCLIP_BENCH_VERBOSE"):
            print(f"[bench rank {rank} +{time.time() - t_start:6.1f}s] {msg}", file=sys.stderr, flush=True)

    from x_clip_b200 import _lib, kernels
    lib = _lib.load()
    _lib.call("xclip_init")
    for kv in filter(None, args.tune.split(",")):
        k, v = kv.split("=")
        lib.xclip_tune_set(int(k), int(v))

    parity = None
    if world > 1 and not args.no_parity:
        parity = multirank_parity(dev, rank, world)
        note(f"multi-rank parity: {parity}")

    model_cfg, _ = WORKLOADS[args.workload]
    B = args.batch
    run = Runner(model_cfg, args.loss, B, args.microbatch, args.patch_dropout, dev, rank, world,
                 grad_sync=args.grad_sync, host_buffers=0 if args.no_e2e else 2, retain=args.retain)
    note("model + data ready")

    # ---- (1) device-resident timing
    for i in range(max(args.warmup, 1)):
        run.step()
        if os.environ.get("XCLIP_BENCH_VERBOSE"):
            torch.cuda.synchronize()
            note(f"warm-up step {i} done, plan {getattr(run.clip, 'last_step_plan', None)}")
    run.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.xclip_launch_count_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    run.barrier()
    e0.record()
    for _ in range(args.steps):
        loss = run.step()
    e1.record()
    run.barrier()
    ms_dev = run.max_over_ranks(e0.elapsed_time(e1))
    launches = lib.xclip_launch_count()
    last_loss = loss.item()
    plan = getattr(run.clip, "last_step_plan", None) if args.microbatch else None
    peak_mem = torch.cuda.max_memory_allocated(dev)
    clocks = sampler.stop() if rank == 0 else None
    note(f"device-resident timing done: {ms_dev / args.steps:.1f} ms/step")
    if args.dump_outputs and rank == 0:
        import numpy as np
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        for name, arr in step_outputs(loss, run.clip).items():
            np.save(out_dir / f"{name}.npy", arr)
        note(f"outputs of the last timed step written to {out_dir}")

    # ---- (2) end-to-end: pinned host -> device copy of every step's batch (side stream, double
    #          buffered) + loss read-back, all inside the timed region
    ms_e2e, h2d_bytes = None, 0
    if not args.no_e2e:
        host = run.host
        h2d_bytes = host[0][0].numel() * 8 + host[0][1].numel() * 4
        copy_stream = torch.cuda.Stream(device=dev)
        slots = [(torch.empty_like(run.text), torch.empty_like(run.image)) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]

        def issue_copy(i):
            s = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[s])
                slots[s][0].copy_(host[s][0], non_blocking=True)
                slots[s][1].copy_(host[s][1], non_blocking=True)
                ready[s].record(copy_stream)

        for s in range(2):
            consumed[s].record(torch.cuda.current_stream())
        # the two device input slots changed the memory picture: one untimed step lets the allocator
        # settle on the new steady state before the timed region
        run.step(slots[0][0].copy_(host[0][0]), slots[0][1].copy_(host[0][1]))
        run.barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        issue_copy(0)
        for i in range(args.steps):
            s = i % 2
            if i + 1 < args.steps:
                issue_copy(i + 1)
            torch.cuda.current_stream().wait_event(ready[s])
            loss = run.step(slots[s][0], slots[s][1])
            consumed[s].record(torch.cuda.current_stream())
            _ = loss.item()                      # device -> host read of the step's result
        f1.record()
        run.barrier()
        ms_e2e = run.max_over_ranks(f0.elapsed_time(f1))
        del slots
        note("e2e timing done")

    # ---- (2b) N > 1: the same step with the weight-gradient all-reduce inside (GradSync buckets
    #           overlapped with backward; the reference leaves this to the user's DDP wrapper)
    with_sync = None
    if world > 1 and not args.grad_sync:
        from x_clip_b200.distributed import GradSync
        run.grad_sync = GradSync(run.clip)
        n_sync = max(2, min(args.steps, 3))
        ms_sync, _ = run.timed(n_sync, 1)
        run.grad_sync.remove()
        run.grad_sync = None
        nbytes = sum(p.numel() * 4 for p in run.params if p.requires_grad)
        with_sync = {"pairs_per_s": round(B * world * n_sync / (ms_sync / 1e3), 2),
                     "ms_per_step": round(ms_sync / n_sync, 3), "steps": n_sync,
                     "allreduced_bytes_per_step": nbytes,
                     "what": "x_clip_b200.distributed.GradSync: fp32 bucketed all-reduce launched from inside backward"}
        note(f"with grad sync: {with_sync}")

    # ---- (3) instrumented step for the roofline (every rank runs it - it contains collectives)
    prof = None
    if not args.no_profile:
        if rank == 0:
            kernels.PROF.start()
        run.step()
        if rank == 0:
            prof = kernels.PROF.stop()
        run.barrier()
        note("profile step done")
    run.close()

    # ---- (4) side measurements on the same GPUs
    extras = None
    if not args.no_extras and args.workload == "cfg3" and args.loss == "nce":
        extras = {}
        for key, (wl, loss_k, b, mb, st) in {
                "cfg2": ("cfg2", "nce", 1024, 0, 5),
                "cfg4_filip": ("cfg2", "filip", 256, 0, 3),
                "cfg5_dcl_extra": ("cfg2", "dcl_extra", 8192, 1024, 2)}.items():
            try:
                r = Runner(WORKLOADS[wl][0], loss_k, b, mb, args.patch_dropout, dev, rank, world)
                ms, l = r.timed(st, 2)
                r.close()
                extras[key] = {"pairs_per_s": round(b * world * st / (ms / 1e3), 1), "ms_per_step": round(ms / st, 2),
                               "pairs_per_gpu": b, "global_batch": b * world, "microbatch": mb or None,
                               "steps": st, "loss": round(l, 5),
                               "model": "README CLIP (cfg1/cfg2 model)", "loss_kind": LOSS_TXT[loss_k]}
            except Exception as e:
                extras[key] = {"error": f"{type(e).__name__}: {str(e)[:160]}"}
                if os.environ.get("XCLIP_BENCH_VERBOSE"):
                    import traceback
                    traceback.print_exc()
                r = None
                torch.cuda.empty_cache()
            note(f"extra {key}: {extras[key]}")

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_burst = peaks.get("bf16_tflops") or 1640.0
    peak_hbm = peaks.get("hbm_gbs") or 6500.0
    peak_src = ("MEASURED_PEAKS.json (bf16_tflops_sustained for kernels inside the step, hbm_gbs)" if peaks
                else "fallback 1.4 PF sustained / 6.5 TB/s (B200_PROFILING.md)")

    roofline, families = None, None
    if prof:
        total_ms = sum(d["ms"] for d in prof.values())
        families = {k: {"calls": d["calls"], "ms": round(d["ms"], 3),
                        "share": round(d["ms"] / total_ms, 4),
                        "tflops": round(d["flops"] / d["ms"] / 1e9, 1) if d["flops"] else None,
                        "gbs": round(d["bytes"] / d["ms"] / 1e6, 1)} for k, d in sorted(prof.items())}
        gem = [prof[k] for k in ("gemm_fwd", "gemm_dgrad", "gemm_wgrad") if k in prof]
        g_ms = sum(d["ms"] for d in gem)
        g_fl = sum(d["flops"] for d in gem)
        g_calls = sum(d["calls"] for d in gem)
        achieved = g_fl / g_ms / 1e9
        traffic = None
        tf = ROOT / "profiles" / "gemm_traffic.json"
        if tf.exists():
            ratio = json.loads(tf.read_text()).get("traffic_over_algorithmic")
            if ratio:
                traffic = round(ratio * sum(d["bytes"] for d in gem) / g_calls)
        roofline = {"kernel": "gemm_pair_kernel / gemm_bf16_kernel (tcgen05, plain-epilogue fwd+dgrad+wgrad launches; "
                              "the fused feed-forward GEMMs are listed under feed_forward_fused)",
                    "bound": "tensor", "achieved": round(achieved, 1), "peak": peak_tf,
                    "unit": "TFLOP/s", "frac": round(achieved / peak_tf, 4),
                    "frac_of_burst_peak": round(achieved / peak_burst, 4), "traffic": traffic,
                    "traffic_note": "ncu dram bytes / algorithmic bytes ratio (profiles/gemm_traffic.json) x live algorithmic bytes per launch",
                    "peak_source": peak_src, "launches_per_step": g_calls,
                    "avg_launch_ms": round(g_ms / g_calls, 4),
                    "flops_per_launch": g_fl / g_calls,
                    "algorithmic_bytes_per_launch": round(sum(d["bytes"] for d in gem) / g_calls),
                    "share_of_step": round(g_ms / total_ms, 4)}

        def sub(names, label, note_txt):
            ds = [prof[k] for k in names if k in prof]
            if not ds:
                return None
            ms = sum(d["ms"] for d in ds); fl = sum(d["flops"] for d in ds); by = sum(d["bytes"] for d in ds)
            tfs, gbs = fl / ms / 1e9, by / ms / 1e6
            # the binding roofline is whichever fraction is larger
            ft, fh = tfs / peak_burst, gbs / peak_hbm
            return {"kernel": label, "launches_per_step": sum(d["calls"] for d in ds), "ms_per_step": round(ms, 3),
                    "share_of_step": round(ms / total_ms, 4), "tflops": round(tfs, 1),
                    "tensor_frac_of_burst_peak": round(ft, 4), "hbm_gbs": round(gbs, 1),
                    "hbm_frac_of_peak": round(fh, 4), "bound": "hbm" if fh > ft else "tensor",
                    "frac": round(max(ft, fh), 4), "note": note_txt}
        roofline["feed_forward_fused"] = {
            "up": sub(["ff_up"], "gemm_pair_kernel<PEPI_FF_UP> (up-projection GEMM + GEGLU epilogue)",
                      "flops = the GEMM only (2*M*8d*d); the epilogue also evaluates 4d GELUs per token and writes "
                      "u (8d, skipped in forward-only sweeps) + hp (4d)"),
            "down": sub(["ff_down"], "gemm_pair_kernel<PEPI_FF_DOWN> (down-projection GEMM + LayerNorm fold + residual)",
                        "flops = the GEMM only (2*M*4d*d)"),
            "bwd": sub(["ff_bwd"], "gemm_pair_kernel<PEPI_FF_BWD2> (dgrad GEMM + LayerNorm/GEGLU backward epilogue, u by TMA one and a half steps ahead)",
                       "flops = the GEMM only (2*M*4d*d); reads u 8d, writes du 8d: HBM-bound by design")}
        roofline["attention"] = {
            "fwd": sub(["attn_fwd"], "attn_fwd_small_kernel / attn_fwd_wg_kernel",
                       "algorithmic: 4 n^2 64 flops and q,k,v read + o write per (batch, head); at n = 98 / 78 "
                       "(cfg3) the arithmetic intensity is n/2 ~ 40-50 flop/B, below the B200 ridge (~250): "
                       "short-sequence attention is HBM-bound, 40 % of the tensor peak is not reachable"),
            "bwd": sub(["attn_bwd"], "attn_delta_kernel + attn_bwd_small_kernel / attn_bwd_kernel",
                       "algorithmic: 10 n^2 64 flops; q,k,v,o,dO read + dq,dk,dv write")}
        roofline["logits"] = {
            "fwd": sub(["nce_fwd"], "gemm_bf16_kernel<EPI_NCE_FWD> + nce_finalize_kernel",
                       "S never materialised: tensor-bound by design (3.6k flop/B at cfg3, SURVEY 8d); split-bf16 "
                       "operands make the contraction 3x the nominal 2*B_l*B_g*D flops (counted)"),
            "bwd": sub(["nce_bwd"], "gemm_bf16_kernel<EPI_NCE_BWD>", "writes bf16 g[B_l, B_g] once")}

    cpu_baseline, eager = None, None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_rate(model_cfg, LOSS_KW[args.loss], args.patch_dropout, 8, steps=20, warmup=1, budget_s=25.0)
        cpu_baseline = {"value": round(r["value"], 3), "unit": "pairs/s", "cores": r["cores"], "kind": r["kind"],
                        "sample": f"{r['steps']} steps of {r['batch']} pairs of the same model (fwd+bwd, fp32, "
                                  f"patch dropout {args.patch_dropout}), {r['ms']:.0f} ms/step"}
        r1 = cpu_reference_rate(README_CFG, {}, 0.5, 4, steps=10, warmup=1, budget_s=10.0)
        cpu_baseline["cfg1_readme_batch4"] = {"value": round(r1["value"], 3), "ms_per_step": round(r1["ms"], 1),
                                              "kind": r1["kind"], "cores": r1["cores"]}
    if world == 1 and not args.no_eager_baseline:
        eager = gpu_eager_baseline(model_cfg, LOSS_KW[args.loss], args.patch_dropout, dev)

    Bg = B * world
    line = {
        "metric": METRIC, "value": round(Bg * args.steps / (ms_dev / 1e3), 2), "unit": "pairs/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_dev / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_text(args, plan=plan), "global_batch": Bg,
                   "global_batch_at_8_gpus": B * 8,
                   "step_plan": plan, "peak_hbm_bytes_allocated": int(peak_mem),
                   "parallelism": f"dp{world}" + ("+grad-allreduce" if args.grad_sync and world > 1 else ""),
                   "l2": "per-step working set (tens of GB of activations) >> 126 MB L2; no flush needed",
                   "timing": "CUDA events on the launching stream, barrier+synchronize both sides, max over ranks",
                   "loss": round(last_loss, 5)},
        "clocks": clocks,
        "e2e": None if ms_e2e is None else {
            "value": round(Bg * args.steps / (ms_e2e / 1e3), 2), "unit": "pairs/s",
            "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
            "ms_per_step": round(ms_e2e / args.steps, 3)},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "gpu_eager_baseline": eager,
        "multirank_parity": parity,
        "with_grad_sync": with_sync,
        "other_workloads": extras,
        "kernel_families": families,
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
