"""Variable-length batches in the graphed bf16 KD step at bench.py's configuration (B 512, V 5000, E 256, H 512, L 2), one JSON line.

The reference's loader pads every batch to its own longest caption.  GraphedKDStep(max_steps=T_cap) captures one graph with a device
step count and replays it for any T <= T_cap; this measures what that costs next to a graph captured at exactly T:
  * varlen_ms[T]   the max_steps graph (T_cap = --cap) replayed on batches of T steps
  * fixed_ms[T]    a graph captured at exactly T (max_steps=None), the same batch
  * eager_ms[T]    the same step issued eagerly (no graph), at the first T only, for scale
  * loss[...][T]   out5 of the last timed step of each (the variable graph and the fixed graph of one T start from the same weights)
  * gpu / power_limit_w from the same process
Each time: CUDA events around --steps replays after --warmup (eval mode: no dropout).  Every step is an optimizer step, so the
loss drifts a little over the timed window; the losses are reported, not compared."""
import argparse
import json
import os
import subprocess
import sys

import torch


def build(cfg, dev, T, max_steps, use_graph=True):
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    from imagecaptioner_b200.optim import FlatAdamW, reference_param_groups
    from oracle import kd_oracle as O
    from tests.harness import build_student
    import bench
    V, E, H, L = cfg["V"], cfg["E"], cfg["H"], cfg["L"]
    model, projector = build_student(O.init_student_params(V, E, H, L, True, seed=0), O.init_projector_params(cfg["Et"], E, seed=1),
                                     V, E, H, L, True, cfg["Et"], dev)
    model.decoder.compute_dtype = torch.bfloat16
    opt = FlatAdamW(reference_param_groups(model, projector, 1e-4), weight_decay=0.01, max_grad_norm=1.0, single_process=True)
    batch = {k: v.to(dev) for k, v in bench.make_batch(dict(cfg, T=T), 1234).items()}
    kd = GraphedKDStep(model, projector, DistillationLoss(0.7, 0.2, 0.1, 4.0, vocab_size=V), opt, None, batch, max_grad_norm=1.0,
                       autocast_dtype=torch.bfloat16, use_graph=use_graph, warmup_steps=3, max_steps=max_steps)
    return kd, batch


def timed(kd, steps, warmup):
    for _ in range(warmup):
        kd.step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        out5 = kd.step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, out5.tolist()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cap", type=int, default=32)
    ap.add_argument("--lengths", default="32,20,12")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    assert torch.cuda.is_available(), "bench_varlen needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    cfg = dict(bench.CFG)
    lengths = [int(t) for t in args.lengths.split(",")]
    out = {"gpu": torch.cuda.get_device_name(dev), "power_limit_w": pl, "config": dict(cfg, T=None), "cap": args.cap,
           "steps": args.steps, "warmup": args.warmup, "varlen_ms": {}, "fixed_ms": {}, "eager_ms": {}, "loss": {"varlen": {}, "fixed": {}, "eager": {}}}
    kd, _ = build(cfg, dev, lengths[0], args.cap)
    for T in lengths:
        batch = {k: v.to(dev) for k, v in bench.make_batch(dict(cfg, T=T), 1234).items()}
        kd.load(batch, non_blocking=False)
        out["varlen_ms"][T], out["loss"]["varlen"][T] = timed(kd, args.steps, args.warmup)
    del kd
    torch.cuda.empty_cache()
    for T in lengths:
        kd, _ = build(cfg, dev, T, None)
        out["fixed_ms"][T], out["loss"]["fixed"][T] = timed(kd, args.steps, args.warmup)
        del kd
        torch.cuda.empty_cache()
    T = lengths[0]
    kd, _ = build(cfg, dev, T, None, use_graph=False)
    out["eager_ms"][T], out["loss"]["eager"][T] = timed(kd, max(3, args.steps // 5), 2)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
