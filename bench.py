#!/usr/bin/env python
"""KD train-step throughput of the B200-native hot path (BASELINE.json metric: KD train samples/sec).

One "step" = one pass of the hot path over one synthetic batch, replaying the reference's training step
(src/train_student_kd.py:262-303) with the encoders outside the path: refinement + attention-LSTM decoder
forward, FeatureProjector, DistillationLoss (all four terms), backward to every decoder / refinement /
projector parameter and the encoder features, gradient all-reduce (N>1), two-group global-norm clip and AdamW.

  python bench.py [--gpus N] [--steps K] [--warmup W]              # our arm  (torchrun launches N>1)
  python bench.py --impl reference ...                             # the reference algorithm on the host CPU cores
  torchrun ... bench.py --gpus N --check                           # N-rank step == 1-GPU step on the concatenated batch (fp32)
  python bench.py ... --dump-outputs DIR                           # also write what the last timed step returned, DIR/loss.npy

Prints ONE JSON line (rank 0).  `value` = samples/s with inputs resident in HBM in the parity configuration (eval mode, dropout
off: the configuration every parity test and the CPU / GPU baselines run, and round 1's headline); `value_dropout` = the same step
in the reference's training mode (dropout 0.3 decoder, 0.1 refinement, 0.1 projector; SURVEY.md section 8d "p=0.3 for throughput
runs"; a fresh mask per graph replay); `e2e` = the step through the public modules with every step's inputs copied from pinned
host memory and the loss read back.  `legs` carries BASELINE configs[3] (greedy decode) and configs[4]
(large variant, 32 and 256 per GPU); `gpu_eager_baseline` the stock torch.nn path on the same GPU; `cpu_baseline` the oracle
port on the host cores at the SAME batch size.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# BASELINE.json configs[1]: default student, batch 512 per GPU, len 20, vocab 5000, ViT-small teacher features 197x384
CFG = dict(B=512, T=20, V=5000, E=256, H=512, L=2, S=49, St=197, Et=384)
# BASELINE.json configs[4]: large variant (README.md:188-195), ViT-small teacher features are 384-d = E: identity channel projection
CFG_LARGE = dict(B=32, T=20, V=10000, E=384, H=768, L=3, S=49, St=197, Et=384)
DROPOUT = 0.3            # src/train_student_kd.py:175-182 builds the student with dropout=0.3
METRIC = "kd_train_samples_per_sec"


def log(msg):
    if os.environ.get("BENCH_VERBOSE"):
        print(f"[bench rank {os.environ.get('RANK', '0')} +{time.perf_counter() - T0:7.2f}s] {msg}", file=sys.stderr, flush=True)


T0 = time.perf_counter()


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


def fwd_flops(cfg, B, T, train):
    """Algorithmic FLOPs of the decoder path (SURVEY.md section 8d): per token 2HE + 2(2E)E + sum_l 8H(in_l+H) + 2HE + 2EV, plus
    2*S*E^2 per sequence for the hoisted attention projection; training = 3x forward."""
    E, H, L, V, S = cfg["E"], cfg["H"], cfg["L"], cfg["V"], cfg["S"]
    tok = 2 * H * E + 2 * (2 * E) * E + sum(8 * H * ((E if k == 0 else H) + H) for k in range(L)) + 2 * H * E + 2 * E * V
    return (3 if train else 1) * (B * T * tok + B * 2 * S * E * E)


class ClockSampler:
    """SM clock / throttle reasons DURING the measurement, polled in-process through NVML every 5 ms from before the warm-up
    until the timed region ends (an nvidia-smi subprocess does not even start inside a 50 ms timed region)."""

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.thread, self.err = index, [], False, None, None
        self.mark = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self.stop_flag:
                    try:
                        self.rows.append((time.perf_counter(), float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), int(get_reasons(h))))
                    except Exception as exc:          # keep sampling; report the last error
                        self.err = repr(exc)
                    time.sleep(0.005)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
        except Exception as exc:
            self.err = repr(exc)

    def mark_timed(self, t0, t1):
        self.mark = (t0, t1)

    def stop(self):
        self.stop_flag = True
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + str(self.err)], "samples": 0}
        self.thread.join(timeout=1.0)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        rows = self.rows
        timed = [r for r in rows if self.mark and self.mark[0] <= r[0] <= self.mark[1]]
        use = timed if len(timed) >= 3 else rows
        reasons = sorted({name for r in use for name, b in bits.items() if r[2] & b})
        return {"sm_mhz": statistics.median(r[1] for r in use) if use else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(rows), "samples_in_timed_region": len(timed), "source": "NVML in-process, 5 ms period, warm-up + timed region"}


def make_batch(cfg, seed):
    from oracle import kd_oracle as O   # synthetic-input generator shared with the tests (data only, no compute)
    return O.synthetic_batch(cfg["B"], cfg["T"], cfg["V"], cfg["E"], cfg["H"], cfg["S"], cfg["St"], cfg["Et"], seed=seed)


def workload_config(n, B=None):
    B = CFG["B"] if B is None else B
    return {"workload": "BASELINE configs[1]: CaptioningStudent default (E256 H512 2-layer LSTM, 49x256 feats, refinement) KD train step, "
                        f"batch {B}/GPU, len 20, vocab 5000, synthetic ViT-small teacher logits + 197x384 features + hidden states, bf16 compute / fp32 master",
            "per_gpu_batch": B, "global_batch": B * n, "seq_len": CFG["T"], "vocab": CFG["V"], "parallelism": f"dp{n}",
            "step": "refinement+decoder fwd, projector, 4-term KD loss, bwd, grad allreduce, clip, AdamW",
            "l2_policy": "inputs per step (~410 MB logits+teacher) exceed the 126 MB L2; no explicit flush"}


# ---------------------------------------------------------------------------------------------- CPU: the oracle port
class CpuStep:
    """The reference algorithm (oracle port: plain tensor arithmetic + autograd on the host cores) for the same step, with the
    reference's optimizer block: three AdamW LR groups, clip_grad_norm_ on the student and on the projector (src/train_student_kd.py:219-234, :290-303).
    fp32, eval mode (BASELINE.md section 3)."""

    def __init__(self, B):
        from oracle import kd_oracle as O
        self.O, self.cfg = O, dict(CFG, B=B)
        cfg = self.cfg
        params = O.init_student_params(cfg["V"], cfg["E"], cfg["H"], cfg["L"], True, seed=0)
        pparams = O.init_projector_params(cfg["Et"], cfg["E"], seed=1)
        self.batch = make_batch(cfg, 1234)
        self.P = {k: v.clone().requires_grad_(True) for k, v in params.items()}
        self.Q = {k: v.clone().requires_grad_(True) for k, v in pparams.items()}
        dec = [v for k, v in self.P.items() if k.startswith("decoder.")]
        other = [v for k, v in self.P.items() if not k.startswith("decoder.")] + list(self.Q.values())
        self.opt = torch.optim.AdamW([{"params": dec, "lr": 1e-4}, {"params": other, "lr": 1e-4}], lr=1e-4, weight_decay=0.01)

    def __call__(self):
        O, cfg, batch = self.O, self.cfg, self.batch
        feats = batch["encoder_features"].clone().requires_grad_(True)
        outputs, enc, hids, _ = O.student_forward(self.P, feats, batch["captions_input"], True)
        tproj = O.feature_projector(self.Q, batch["teacher_features"], cfg["S"])
        th = batch["teacher_hiddens"]
        total, _ = O.distillation_loss({"logits": outputs, "encoder_features": enc, "hidden_states": hids},
                                       {"logits": batch["teacher_logits"], "encoder_features": tproj,
                                        "hidden_states": [th[t] for t in range(th.shape[0])]}, batch["targets"])
        self.opt.zero_grad(set_to_none=True)
        total.backward()
        torch.nn.utils.clip_grad_norm_(list(self.P.values()), 1.0)
        torch.nn.utils.clip_grad_norm_(list(self.Q.values()), 1.0)
        self.opt.step()
        return float(total.detach())


def run_reference(args):
    """--impl reference: the oracle port on all host cores, at the configuration's OWN batch size (B = 512) when the requested
    steps fit a ~4 minute budget (a step is ~4-6 s), else at the largest power-of-two batch that does; the line says which."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    budget = float(os.environ.get("B2C_REF_BUDGET_S", "240"))
    B = CFG["B"]
    step = CpuStep(B)
    t0 = time.perf_counter(); step(); first = time.perf_counter() - t0
    while B > 16 and first * (args.steps + args.warmup) > budget:
        B //= 2
        step = CpuStep(B)
        t0 = time.perf_counter(); step(); first = time.perf_counter() - t0
    for _ in range(max(args.warmup - 1, 0)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = B / dt
    sample = (f"{args.steps} whole KD steps (fwd + 4-term loss + bwd + 2 clip norms + AdamW) at B={B}"
              f"{'' if B == CFG['B'] else ' (reduced from 512 to fit the time budget; per-sample rate)'}, T=20 V=5000, fp32, eval mode, oracle port, {threads} threads")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus, B), "batch_run": B,
            "cpu_baseline": {"value": val, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_baseline(budget_s=25.0):
    """Oracle port on the host cores inside our own run (rank 0, N=1 only): bounded sample at the benchmark's batch size B=512
    (a few steps, ~20-30 s), plus the reference loader's own batch (16, src/data_loader.py:120-121) as an extra key."""
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    out = {}
    for B, budget, cap in ((CFG["B"], budget_s, 6), (16, 4.0, 20)):
        step = CpuStep(B)
        step()                                                  # warm-up
        t0, n = time.perf_counter(), 0
        while n < 2 or (time.perf_counter() - t0 < budget and n < cap):
            step(); n += 1
        dt = (time.perf_counter() - t0) / n
        out[B] = (B / dt, n)
    v, n = out[CFG["B"]]
    return {"value": v, "unit": "samples/s", "cores": threads, "kind": "port",
            "sample": f"{n} whole KD steps (fwd + loss + bwd + clip + AdamW) at B={CFG['B']} T=20 V=5000 fp32 eval mode with the oracle port, {threads} threads",
            "value_b16": out[16][0], "sample_b16": f"{out[16][1]} steps at B=16 (BASELINE configs[0]); per-sample rate"}


# ---------------------------------------------------------------------------------------------- GPU: stock torch.nn path
def gpu_eager_baseline(dev, steps=5):
    """The "existing Blackwell path" (SURVEY.md section 2.1): the same step with the stock torch.nn modules the reference
    composes (cuDNN LSTM stepped per token, cuBLAS, ATen element-wise), eager, on the same GPU: fp32 and under autocast."""
    from oracle import kd_oracle as O, eager_torch as ET
    cfg = CFG
    params = O.init_student_params(cfg["V"], cfg["E"], cfg["H"], cfg["L"], True, seed=0)
    pparams = O.init_projector_params(cfg["Et"], cfg["E"], seed=1)
    batch = {k: (v.to(dev) if v is not None else None) for k, v in make_batch(cfg, 1234).items()}
    out = {"what": "oracle/eager_torch.py: stock nn.LSTM / nn.MultiheadAttention / nn.Linear / F.kl_div ... (the reference's composition), eager, "
                   "fwd + loss + bwd + 2 clip_grad_norm_ + torch.optim.AdamW, B=512 T=20 V=5000, eval mode", "unit": "samples/s"}
    for name, ac in (("fp32", None), ("bf16_autocast", torch.bfloat16), ("fp16_autocast", torch.float16)):
        model, proj = ET.build(params, pparams, cfg["V"], cfg["E"], cfg["H"], cfg["L"], True, cfg["Et"], cfg["S"], dev)
        dec = list(model.decoder.parameters())
        other = list(model.attention_refinement.parameters()) + list(proj.parameters())
        opt = torch.optim.AdamW([{"params": dec}, {"params": other}], lr=1e-4, weight_decay=0.01)

        scaler = torch.amp.GradScaler("cuda", enabled=(ac == torch.float16))     # the reference's own loop: fp16 autocast + GradScaler

        def step():
            opt.zero_grad(set_to_none=True)
            scaler.scale(ET.kd_loss(model, proj, batch, ac)).backward()
            scaler.unscale_(opt)
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            torch.nn.utils.clip_grad_norm_(proj.parameters(), 1.0)
            scaler.step(opt)
            scaler.update()
        for _ in range(2):
            step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(steps):
            step()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"ms_per_step": ms, "value": cfg["B"] / ms * 1e3}
    return out


# ---------------------------------------------------------------------------------------------- our arm (GPU)
def build_step(cfg, dev, rank, train_mode, dtype=torch.bfloat16, use_graph=True, torch_optimizer=False, single_process=False, seed=1234):
    """model + projector + loss + FlatAdamW + GraphedKDStep over resident synthetic inputs of `cfg`."""
    from imagecaptioner_b200.ddp import FlatGradAllReducer, attach_loss_group
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    from imagecaptioner_b200.optim import FlatAdamW, reference_param_groups
    from oracle import kd_oracle as O
    from tests.harness import build_student
    B, T, V, E, H, L = cfg["B"], cfg["T"], cfg["V"], cfg["E"], cfg["H"], cfg["L"]
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(cfg["Et"], E, seed=1)
    model, projector = build_student(params, pparams, V, E, H, L, True, cfg["Et"], dev, dropout=DROPOUT if train_mode else 0.0)
    if train_mode:
        model.train(); projector.train()
    model.decoder.compute_dtype = dtype
    loss_mod = DistillationLoss(0.7, 0.2, 0.1, 4.0, vocab_size=V)
    if not single_process:
        attach_loss_group(loss_mod)
    if torch_optimizer:                 # A/B: torch's fused AdamW + one global-norm clip instead of the native flat-buffer step
        trainable = [p for p in list(model.parameters()) + list(projector.parameters()) if p.requires_grad]
        reducer = FlatGradAllReducer(trainable, single_process=single_process)
        opt = torch.optim.AdamW(trainable, lr=1e-4, weight_decay=0.01, fused=True, capturable=use_graph)
    else:                               # the reference's LR groups + two clip groups (train_student_kd.py:219-234, :293-297)
        opt = FlatAdamW(reference_param_groups(model, projector, 1e-4), weight_decay=0.01, max_grad_norm=1.0, single_process=single_process)
        reducer = opt.reducer
    host = make_batch(cfg, seed + rank)
    keys = list(GraphedKDStep.INPUT_KEYS)
    pinned = {k: host[k].pin_memory() for k in keys}
    resident = {k: pinned[k].to(dev, non_blocking=True) for k in keys}
    torch.cuda.synchronize()
    kd = GraphedKDStep(model, projector, loss_mod, opt, reducer, resident, max_grad_norm=1.0,
                       autocast_dtype=torch.bfloat16 if dtype == torch.bfloat16 else None, use_graph=use_graph, warmup_steps=3)
    return kd, model, projector, opt, pinned, resident


def time_steps(kd, steps, warmup, barrier_sync, world, dev, sampler=None):
    import torch.distributed as dist
    for _ in range(warmup):
        kd.step()
    barrier_sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier_sync()
    t_a = time.perf_counter()
    ev0.record()
    for _ in range(steps):
        out5 = kd.step()
    ev1.record()
    barrier_sync()
    if sampler is not None:
        sampler.mark_timed(t_a, time.perf_counter())
    tmax = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    return float(tmax.item()) / steps, out5.tolist()


def dump_outputs(out_dir, kd):
    """--dump-outputs: what the last timed KD step returned to its caller, DIR/loss.npy (float32 [total, ce, token_kd, feature_kd,
    hidden_kd]).  Inputs and initial weights are seeded; two runs of one build with the same arguments on a B200 (1000 W power limit)
    agreed to 2.2e-7 relative after 38 steps (--steps 30 --warmup 5) and to 5e-6 after 123 (--steps 100 --warmup 20).  The step's
    parameter gradients, and through AdamW the updated weights, are not written: the K-split GEMM reductions add fp32 partial tiles
    atomically in a run-dependent order, and AdamW turns the resulting last-bit differences of near-zero gradients into +-lr updates,
    so those arrays differ between two runs of one build by far more than rounding."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), kd.out5.detach().float().cpu().numpy())


def run_ours(args):
    import torch.distributed as dist
    from imagecaptioner_b200 import _ops
    from imagecaptioner_b200.graph import GraphedKDStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun for N>1"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    log(f"start world={world} local={local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        log("process group up")
    lib = _ops.load_library()
    cfg = CFG
    B = cfg["B"]
    warmup = max(args.warmup, 3)
    sampler = ClockSampler(local)            # started before anything is warmed up; rank 0 reports
    if rank == 0:
        sampler.start()

    def barrier_sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: the whole step (fwd, loss, bwd, all-reduce, clip, AdamW) as ONE CUDA graph over static, HBM-resident inputs,
    # training mode (dropout 0.3 / 0.1 / 0.1 like the reference's loop; a fresh mask per replay through the device-side counter)
    n_before = lib.b2c_launch_count()
    kd, model, projector, opt, pinned, resident = build_step(cfg, dev, rank, train_mode=args.train_mode, use_graph=not args.no_graph,
                                                             torch_optimizer=args.torch_optimizer)
    launches_per_step = None if args.no_graph else (lib.b2c_launch_count() - n_before) // 4      # 3 warm-up bodies + 1 captured body
    log("step object ready (warm-up + capture done)")
    n0 = lib.b2c_launch_count()
    ms_step, final_loss = time_steps(kd, args.steps, warmup, barrier_sync, world, dev, sampler if rank == 0 else None)
    if launches_per_step is None:
        launches_per_step = (lib.b2c_launch_count() - n0) / (args.steps + warmup)
    value = B * world / (ms_step * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    log(f"value leg done: {ms_step:.3f} ms/step")
    if args.dump_outputs and rank == 0:          # before the e2e leg below takes further steps on the same weights
        dump_outputs(args.dump_outputs, kd)

    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms_step, "value": value, "gpu_launches_per_step": launches_per_step}), flush=True)
        finish(world)
        return

    # ---- e2e: every step's inputs come from pinned host memory (uploaded on a copy stream into a staging set while the
    # previous step computes, then moved device-to-device into the graph's static buffers); the loss goes back to the host
    keys = list(GraphedKDStep.INPUT_KEYS)
    h2d_bytes = sum(pinned[k].numel() * pinned[k].element_size() for k in keys)
    loss_host = torch.zeros(5, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream()
    staging = {k: torch.empty_like(resident[k]) for k in keys}
    staged_evt, consumed_evt = torch.cuda.Event(), torch.cuda.Event()

    def upload():
        copy_stream.wait_event(consumed_evt)
        with torch.cuda.stream(copy_stream):
            for k in keys:
                staging[k].copy_(pinned[k], non_blocking=True)
            staged_evt.record(copy_stream)

    def e2e_loop(n):
        consumed_evt.record()
        upload()
        for i in range(n):
            torch.cuda.current_stream().wait_event(staged_evt)
            kd.load(staging)
            consumed_evt.record()
            if i + 1 < n:
                upload()                                               # next step's H2D overlaps this step's compute
            o5 = kd.step()
            loss_host.copy_(o5, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_loop(2)
    barrier_sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    e2e_loop(args.steps)
    ev1.record()
    barrier_sync()
    e_ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
    e2e_ms = float(e_ms.item()) / args.steps
    e2e_val = B * world / (e2e_ms * 1e-3)
    log("e2e leg done")

    # ---- the same step in the reference's training mode (dropout 0.3 / 0.1 / 0.1, fresh mask per replay), resident inputs
    value_drop = ms_drop = None
    if not args.train_mode and not args.quick:
        kd2, *_ = build_step(cfg, dev, rank, train_mode=True, use_graph=not args.no_graph, torch_optimizer=args.torch_optimizer)
        ms_drop, _ = time_steps(kd2, args.steps, warmup, barrier_sync, world, dev)
        value_drop = B * world / (ms_drop * 1e-3)
        del kd2
        log(f"dropout leg done: {ms_drop:.3f} ms/step")

    peaks = read_peaks()
    roof, extra, legs, eager = None, {}, None, None
    if rank == 0:
        roof, extra = kernel_rooflines(lib, _ops, dev, cfg, peaks)
        if world == 1 and not args.quick:
            legs = {"decode_b2048_len30": decode_leg(dev, peaks, steps=5)}
            for Bl in (32, 256):
                legs[f"large_variant_b{Bl}"] = large_variant_leg(dev, Bl, peaks, steps=max(10, min(args.steps, 30)))
            legs["validation_b512"] = validation_leg(dev, peaks)
            eager = gpu_eager_baseline(dev)
    mode = f"training mode (dropout {DROPOUT} decoder, 0.1 refinement, 0.1 projector; fresh mask per replay)" if args.train_mode else "eval mode (dropout off): the parity configuration"
    line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup if args.warmup >= 3 else warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": workload_config(world), "mode": mode, "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 20, "ms_per_step": e2e_ms,
                    "h2d_gbs_per_rank": h2d_bytes / (e2e_ms * 1e-3) / 1e9},
            "value_dropout": value_drop, "ms_per_step_dropout": ms_drop,
            "gpu_launches": int(launches_per_step * args.steps), "gpu_launches_per_step": launches_per_step, "cuda_graph": not args.no_graph,
            "optimizer": "torch fused AdamW + global clip" if args.torch_optimizer else "native b2c_optimizer_step (3 LR groups, 2 clip groups)",
            "roofline": roof, "kernels": extra, "legs": legs, "gpu_eager_baseline": eager, "loss": final_loss}
    if rank == 0:
        line["cpu_baseline"] = cpu_baseline() if world == 1 and not args.no_cpu_baseline and not args.quick else None
        print(json.dumps(line), flush=True)
    finish(world)


def finish(world):
    """Multi-rank teardown: barrier, flush, hard exit.  destroy_process_group() after CUDA-graph work has been seen to
    block for minutes on this stack (round 1, 2 GPUs: the JSON line was printed, then the job hung until the box timeout)."""
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


# ---------------------------------------------------------------------------------------------- legs of the default line
def decode_leg(dev, peaks, steps=5):
    """BASELINE configs[3]: greedy caption decode, batch 2048, max length 30 (one device-side decode per step of this leg):
    bf16 throughput mode and fp32 token-id-parity mode; bf16-vs-fp32 token agreement; roofline = algorithmic forward FLOPs."""
    from oracle import kd_oracle as O
    from tests.harness import build_student
    V, E, H, L, B, max_len = CFG["V"], CFG["E"], CFG["H"], CFG["L"], 2048, 30
    params = O.init_student_params(V, E, H, L, False, seed=0, logit_scale=8.0)
    model, _ = build_student(params, {}, V, E, H, L, False, E, dev)
    feats = torch.randn(B, CFG["S"], E, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    fl = fwd_flops(CFG, B, max_len, train=False)
    out = {"workload": "BASELINE configs[3]: greedy decode batch 2048, max len 30, default student (no refinement), CUDA-graph replay per decode"}
    toks = {}
    for name, dt in (("bf16", torch.bfloat16), ("fp32", torch.float32)):
        model.decoder.compute_dtype = dt
        for _ in range(3):
            model.decoder.greedy(feats, max_len)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(steps):
            toks[name], lens = model.decoder.greedy(feats, max_len)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"ms_per_decode": ms, "captions_per_s": B / ms * 1e3, "tokens_per_s": B * max_len / ms * 1e3,
                     "roofline": {"bound": "tensor", "achieved": fl / (ms * 1e-3) / 1e12, "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                                  "frac": fl / (ms * 1e-3) / 1e12 / peaks["tf_burst"], "algorithmic_flops": fl}}
    # how far bf16 decoding drifts from the fp32 (token-id parity) decode of the same weights: first-token agreement is the
    # per-step argmax agreement, whole-caption agreement compounds it over 30 autoregressive steps
    same = (toks["bf16"] == toks["fp32"])
    out["bf16_vs_fp32"] = {"first_token_agreement": float(same[0].float().mean()), "all_tokens_agreement": float(same.float().mean()),
                           "captions_identical": float(same.all(dim=0).float().mean())}
    return out


def large_variant_leg(dev, B, peaks, steps):
    """BASELINE configs[4]: E384 H768 3-layer LSTM, V10000, refinement (head_dim 96), identity channel projection 384 -> 384,
    global batch 256 on 8 GPUs = 32 per GPU (and 256 per GPU): the whole KD step in training mode, CUDA-graph replay."""
    cfg = dict(CFG_LARGE, B=B)
    kd, *_ = build_step(cfg, dev, 0, train_mode=True, single_process=True, seed=4321)
    ms, loss = time_steps(kd, steps, 5, torch.cuda.synchronize, 1, dev)
    fl = fwd_flops(cfg, B, cfg["T"], train=True)
    return {"workload": f"BASELINE configs[4]: large variant E384 H768 L3 V10000 + refinement, batch {B}/GPU, len 20, KD train step, training mode",
            "ms_per_step": ms, "samples_per_s": B / ms * 1e3, "loss": loss[0],
            "roofline": {"bound": "tensor", "achieved": fl / (ms * 1e-3) / 1e12, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                         "frac": fl / (ms * 1e-3) / 1e12 / peaks["tf_sustained"], "algorithmic_flops": fl}}


def validation_leg(dev, peaks, steps=10):
    """validate_student_model's per-batch body at BASELINE configs[1] sizes (B=512, T=20, V=5000, bf16): the student forward + the
    loss without gradients + argmax, with the logits materialised (b2c_decoder_forward + b2c_kd_token_eval) and without
    (b2c_decoder_forward_eval: partials in the vocabulary-head GEMM's epilogue; SURVEY.md section 8f row 4)."""
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from oracle import kd_oracle as O
    from tests.harness import build_student
    cfg = CFG
    B, T, V, E, H, L = cfg["B"], cfg["T"], cfg["V"], cfg["E"], cfg["H"], cfg["L"]
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(cfg["Et"], E, seed=1)
    model, projector = build_student(params, pparams, V, E, H, L, True, cfg["Et"], dev)
    model.decoder.compute_dtype = torch.bfloat16
    model.attention_refinement.compute_dtype = torch.bfloat16
    projector.compute_dtype = torch.bfloat16
    batch = {k: (v.to(dev) if v is not None else None) for k, v in make_batch(cfg, 99).items()}
    loss_mod = DistillationLoss(0.7, 0.2, 0.1, 4.0, vocab_size=V)
    out = {"workload": "validate_student_model body, B=512 T=20 V=5000 bf16 (student forward + loss without gradients + argmax), eager launches"}
    with torch.no_grad():
        t_out = {"logits": batch["teacher_logits"], "encoder_features": projector(batch["teacher_features"]), "hidden_states": None}

        def unfused():
            logits, enc, hids, _ = model(batch["encoder_features"], batch["captions_input"])
            return loss_mod.evaluate({"logits": logits, "encoder_features": enc, "hidden_states": hids}, t_out, batch["targets"])[1]

        def fused():
            return loss_mod.evaluate_fused(model, batch["encoder_features"], batch["captions_input"], t_out, batch["targets"])[1]
        for name, fn in (("logits_materialised", unfused), ("logits_free", fused)):
            for _ in range(3):
                d = fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(); e0.record()
            for _ in range(steps):
                d = fn()
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"ms_per_batch": ms, "samples_per_s": B / ms * 1e3, "total_loss": d["total_loss"]}
    out["logits_bytes_not_written_or_read"] = 2 * T * B * V * 2
    return out


def run_decode(args):
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    print(json.dumps(decode_leg(dev, read_peaks(), steps=args.steps)), flush=True)


def kernel_rooflines(lib, _ops, dev, cfg, peaks):
    """Per-kernel achieved bandwidth / FLOP rate: algorithmic bytes (SURVEY.md §8d) / CUDA-event time per launch."""
    B, T, V, E, H = cfg["B"], cfg["T"], cfg["V"], cfg["E"], cfg["H"]
    N = T * B
    y = torch.randn(N, V, device=dev).bfloat16()
    z = torch.randn(N, V, device=dev) * 2
    tgt = torch.randint(1, V, (N,), device=dev)
    nval = torch.tensor([N], dtype=torch.int32, device=dev)
    dy = torch.empty_like(y)
    rows = torch.empty(2, N, device=dev)

    def kd():
        rc = lib.b2c_kd_token_loss(y.data_ptr(), z.data_ptr(), tgt.data_ptr(), N, V, 4.0, 0.7, 0.0, 1.0, nval.data_ptr(), dy.data_ptr(),
                                   rows[0].data_ptr(), rows[1].data_ptr(), _ops.B2C_BF16, torch.cuda.current_stream().cuda_stream)
        assert rc == 0

    def timeit(fn, reps=20):
        """Average device time of one launch: `reps` back-to-back launches captured in a CUDA graph (so the host-side ctypes /
        tensor-map cost of a launch, ~10 us, is not what is measured), timed with CUDA events around 5 replays."""
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                fn()
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (5 * reps) * 1e-3

    t_kd = timeit(kd)
    kd_bytes = N * V * (2 + 4 + 2) + 8 * N                     # read bf16 student + fp32 teacher, write bf16 dlogits, read targets
    traffic, traffic_src = None, None
    for fn in ("r2_kernel_traffic.json", "r1_kernel_traffic.json"):        # dram__bytes_read + write of ONE ncu --set full capture
        tpath = os.path.join(ROOT, "profiles", fn)
        if os.path.exists(tpath):
            rec = json.load(open(tpath)).get("kd_token_loss_pipe_kernel<bf16,3,true>")
            if rec:
                traffic, traffic_src = rec["dram_bytes_read"] + rec["dram_bytes_write"], rec["source"]
                break
    roof = {"kernel": "kd_token_loss_pipe_kernel<bf16,3,true> (b2c_kd_token_loss)", "bound": "hbm", "achieved": kd_bytes / t_kd / 1e9, "peak": peaks["hbm"],
            "unit": "GB/s", "frac": kd_bytes / t_kd / 1e9 / peaks["hbm"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peaks["src"] + " (MEASURED_PEAKS.json hbm_gbs)",
            "algorithmic_bytes_per_launch": kd_bytes, "us_per_launch": t_kd * 1e6}
    # vocabulary head GEMM (time-batched, tcgen05): logits = o1 W2^T, M = T*B, N = V, K = E
    A = torch.randn(N, E, device=dev).bfloat16(); W = torch.randn(V, E, device=dev).bfloat16(); C = torch.empty(N, V, device=dev, dtype=torch.bfloat16)
    t_g = timeit(lambda: _ops.gemm(A, W, N, V, E, C=C))
    fl = 2.0 * N * V * E
    # recurrent gate GEMM of one step (serial part): M = B, N = 4H, K = E+H
    A2 = torch.randn(B, E + H, device=dev).bfloat16(); W2 = torch.randn(4 * H, E + H, device=dev).bfloat16(); C2 = torch.empty(B, 4 * H, device=dev)
    t_g2 = timeit(lambda: _ops.gemm(A2, W2, B, 4 * H, E + H, C=C2))
    fl2 = 2.0 * B * 4 * H * (E + H)
    extra = {"vocab_head_gemm_tcgen05": {"bound": "tensor", "achieved": fl / t_g / 1e12, "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                                         "frac": fl / t_g / 1e12 / peaks["tf_burst"], "us_per_launch": t_g * 1e6, "shape": [N, V, E]},
             "lstm_gate_gemm_tcgen05": {"bound": "tensor", "achieved": fl2 / t_g2 / 1e12, "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                                        "frac": fl2 / t_g2 / 1e12 / peaks["tf_burst"], "us_per_launch": t_g2 * 1e6, "shape": [B, 4 * H, E + H]}}
    return roof, extra


# ---------------------------------------------------------------------------------------------- --check (multi-rank numerics)
def run_check(args):
    """N ranks, each on its shard, against ONE GPU on the concatenated batch, fp32 parity mode, 3 optimizer steps from the same
    initial weights: the averaged all-reduced gradient of step 1, the loss parts and the weights after 3 steps must agree
    (SURVEY.md section 8e: CE divides by the GLOBAL non-PAD count; every other term has equal per-rank denominators).  Run with
    the overlapped exchange (external events around the step graph, deferred weight-gradient join) and with serial collectives.
    One GPU: B2C_FAKE_DP exercises the same control flow with identity collectives (then the reference is the same batch)."""
    import torch.distributed as dist
    from oracle import kd_oracle as O
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = dict(CFG, B=args.check_batch)
    params = O.init_student_params(cfg["V"], cfg["E"], cfg["H"], cfg["L"], True, seed=0)
    pparams = O.init_projector_params(cfg["Et"], cfg["E"], seed=1)

    def reset(model, projector, opt):
        """back to the initial weights and optimizer state (build_step's warm-up + capture bodies already took optimizer steps)"""
        model.load_state_dict({k: v.float() for k, v in params.items()}, strict=False)
        projector.load_state_dict({k: v.float() for k, v in pparams.items()})
        opt.exp_avg.zero_(); opt.exp_avg_sq.zero_(); opt.step_count.zero_()

    def three_steps(kd, opt, scale):
        losses, grad1 = [], None
        for i in range(3):
            o5 = kd.step()
            if i == 0:
                torch.cuda.synchronize()
                grad1 = (opt.reducer.flat * scale).clone()      # multi-rank: the buffer holds the SUM over ranks
            losses.append(o5.clone())
        torch.cuda.synchronize()
        return torch.stack(losses), grad1, opt.flat_param.clone()

    ref = None
    if rank == 0:                              # the 1-GPU run on the concatenated batch
        os.environ.pop("B2C_FAKE_DP", None)
        gcfg = dict(cfg, B=cfg["B"] * world)
        kd1, model1, projector1, opt1, _, _ = build_step(gcfg, dev, 0, train_mode=False, dtype=torch.float32, single_process=True, seed=777)
        shards = [make_batch(cfg, 777 + r) for r in range(world)]
        cat = {k: torch.cat([s[k] for s in shards], dim=0 if k in ("encoder_features", "teacher_features") else 1).to(dev) for k in kd1.static}
        kd1.load(cat)
        reset(model1, projector1, opt1)
        ref = three_steps(kd1, opt1, 1.0)
        offsets = list(zip(opt1.params, opt1.offsets))
        del kd1
    report = {"check": "dp_equals_global_batch", "world": world, "per_rank_batch": cfg["B"], "dtype": "f32", "steps": 3,
              "collectives": "nccl" if world > 1 else "identity (B2C_FAKE_DP, one GPU)"}
    ok_all = True
    for overlap in ("1", "0"):
        os.environ["B2C_OVERLAP_COMM"] = overlap
        if world == 1:
            os.environ["B2C_FAKE_DP"] = "1"
        kd, model, projector, opt, _, _ = build_step(cfg, dev, rank, train_mode=False, dtype=torch.float32, seed=777)
        reset(model, projector, opt)
        losses, grad1, flatw = three_steps(kd, opt, 1.0 / world)
        l0 = losses[0].clone()
        if world > 1:
            dist.all_reduce(l0); l0 /= world
        if rank == 0:
            ref_losses, ref_grad1, ref_w = ref
            seg_err = max(float((grad1[o:o + p.numel()] - ref_grad1[o:o + p.numel()]).abs().max() / (ref_grad1[o:o + p.numel()].abs().max() + 1e-30))
                          for p, o in offsets)
            g_err = float((grad1 - ref_grad1).abs().max() / ref_grad1.abs().max())
            dw = (flatw - ref_w).abs()
            w_err = float(dw.max() / ref_w.abs().max())
            frac_off = float((dw > 1e-5 * ref_w.abs().max()).float().mean())
            # token-KD / feature / hidden parts are means with equal per-rank denominators: their rank average is the global value
            l_err = max(abs(a - b) / max(abs(b), 1e-12) for a, b in zip(l0.tolist()[2:], ref_losses[0].tolist()[2:]))
            entry = {"grad_step1_rel_err_flat": g_err, "grad_step1_rel_err_worst_tensor": seg_err, "weights_after_3_steps_rel_err": w_err,
                     "weights_fraction_beyond_1e-5": frac_off, "loss_parts_rel_err": l_err, "overlapped_exchange": bool(kd.overlap_comm),
                     "loss_global": ref_losses[0].tolist(), "loss_ranks_avg": l0.tolist()}
            # Adam turns a near-zero gradient into a +-lr update, so single elements whose gradient is ~0 may differ between two
            # summation orders; the gradient is the exact check, the weights are held to 1e-5 on all but a 1e-3 fraction of elements
            entry["ok"] = bool(seg_err < 1e-4 and g_err < 1e-5 and l_err < 1e-5 and frac_off < 1e-3)
            ok_all = ok_all and entry["ok"]
            report["overlap_comm_" + overlap] = entry
        del kd
    if rank == 0:
        report["ok"] = ok_all
        print(json.dumps(report), flush=True)
        if args.out:
            with open(args.out, "w") as f:
                json.dump(report, f, indent=1)
    finish(world)
    if rank == 0 and not ok_all:
        sys.exit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b2c", choices=["b2c", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="value + e2e + kernel rooflines only (no legs, no eager / CPU baselines, no dropout-off leg)")
    ap.add_argument("--train-mode", action="store_true", help="time the reference's training mode (dropout on) as the headline instead of the parity configuration")
    ap.add_argument("--workload", default="kd_step", choices=["kd_step", "decode"], help="kd_step = the contract's metric (default); decode = configs[3] greedy decode leg alone")
    ap.add_argument("--torch-optimizer", action="store_true", help="A/B: torch fused AdamW + one global clip instead of the native optimizer step")
    ap.add_argument("--no-graph", action="store_true", help="issue the step eagerly instead of replaying one CUDA graph")
    ap.add_argument("--profile", action="store_true", help="only warm-up + timed steps (for ncu launch lists); prints a reduced line")
    ap.add_argument("--check", action="store_true", help="multi-rank numerics: N-rank step vs 1-GPU step on the concatenated batch (fp32)")
    ap.add_argument("--check-batch", type=int, default=64)
    ap.add_argument("--out", default=None, help="--check: also write the report to this file")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed KD step returned (its five loss parts) as DIR/loss.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.check or args.workload != "kd_step" or args.impl != "b2c"):
        ap.error("--dump-outputs applies to the timed KD step (--impl b2c --workload kd_step, without --check)")
    if args.check:
        run_check(args)
    elif args.workload == "decode":
        run_decode(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
