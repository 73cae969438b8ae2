"""Teacher outputs in fp32 / bf16 / fp16 at bench.py's configuration (B 512, T 20, E 256, H 512, L 2, 197x384 teacher features, bf16
compute, eval mode), at V = 5000 and V = 4999, one JSON line.  The three teacher precisions are built in one process and timed
alternately (--rounds rounds of --steps steps each):
  * step_ms          graphed KD step over resident inputs, CUDA events
  * token_pass       the token KD + CE pass alone: 20 launches of b2c_kd_token_loss_teacher captured in one CUDA graph (as bench.py's
                     roofline leg does), with its compulsory bytes (read y bf16 + z in the teacher's type, write dlogits bf16) and GB/s
  * e2e              bench.py's e2e leg: every step's inputs from pinned host memory on a copy stream into a staging set, then
                     load() + step(); H2D bytes per step, ms per step, samples/s
  * gpu / power_limit_w from the same process."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (CFG, make_batch: the benchmarked workload, unchanged)

TEACHER_KEYS = ("teacher_logits", "teacher_features", "teacher_hiddens")
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def build(cfg, dev, tdt):
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    from imagecaptioner_b200.optim import FlatAdamW, reference_param_groups
    from oracle import kd_oracle as O
    from tests.harness import build_student
    B, T, V, E, H, L = cfg["B"], cfg["T"], cfg["V"], cfg["E"], cfg["H"], cfg["L"]
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(cfg["Et"], E, seed=1)
    model, projector = build_student(params, pparams, V, E, H, L, True, cfg["Et"], dev)
    model.decoder.compute_dtype = torch.bfloat16
    opt = FlatAdamW(reference_param_groups(model, projector, 1e-4), weight_decay=0.01, max_grad_norm=1.0, single_process=True)
    host = bench.make_batch(cfg, 1234)
    pinned = {k: (host[k].to(tdt) if k in TEACHER_KEYS else host[k]).pin_memory() for k in GraphedKDStep.INPUT_KEYS}
    resident = {k: v.to(dev) for k, v in pinned.items()}
    kd = GraphedKDStep(model, projector, DistillationLoss(0.7, 0.2, 0.1, 4.0, vocab_size=V), opt, opt.reducer, resident, max_grad_norm=1.0,
                       autocast_dtype=torch.bfloat16, use_graph=True, warmup_steps=3)
    return kd, pinned, resident


def time_steps(kd, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out5 = kd.step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, out5.tolist()


def e2e(kd, pinned, resident, steps):
    """bench.py's e2e leg: the next step's H2D copy overlaps this step's compute."""
    keys = list(pinned)
    staging = {k: torch.empty_like(resident[k]) for k in keys}
    copy_stream = torch.cuda.Stream()
    staged, consumed = torch.cuda.Event(), torch.cuda.Event()
    loss_host = torch.zeros(5, dtype=torch.float32).pin_memory()

    def upload():
        copy_stream.wait_event(consumed)
        with torch.cuda.stream(copy_stream):
            for k in keys:
                staging[k].copy_(pinned[k], non_blocking=True)
            staged.record(copy_stream)

    def loop(n):
        consumed.record()
        upload()
        for i in range(n):
            torch.cuda.current_stream().wait_event(staged)
            kd.load(staging)
            consumed.record()
            if i + 1 < n:
                upload()
            loss_host.copy_(kd.step(), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    loop(2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loop(steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    h2d = sum(v.numel() * v.element_size() for v in pinned.values())
    return {"h2d_bytes_per_step": h2d, "ms_per_step": ms, "samples_per_s": kd.static["targets"].shape[1] / (ms * 1e-3)}


def token_pass(lib, _ops, dev, V, N, tdt, reps=20):
    """b2c_kd_token_loss_teacher alone, `reps` launches in one CUDA graph: time per launch and bytes/s over its compulsory traffic."""
    Vp = (V + 7) // 8 * 8
    g = torch.Generator(device=dev).manual_seed(0)
    y = torch.randn(N, V, generator=g, device=dev).bfloat16()
    z = (torch.randn(N, V, generator=g, device=dev) * 2).to(tdt)
    t = torch.randint(1, V, (N,), generator=g, device=dev)
    nval = torch.full((1,), N, dtype=torch.int32, device=dev)
    rows = torch.empty(2, N, device=dev)
    dy = torch.empty(N, Vp, dtype=torch.bfloat16, device=dev)
    code = {torch.float32: _ops.B2C_F32, torch.bfloat16: _ops.B2C_BF16, torch.float16: _ops.B2C_F16}[tdt]

    def call():
        rc = lib.b2c_kd_token_loss_teacher(y.data_ptr(), z.data_ptr(), code, t.data_ptr(), N, V, 4.0, 0.7, 0.1, 1.0, nval.data_ptr(),
                                           dy.data_ptr(), Vp, rows[0].data_ptr(), rows[1].data_ptr(), _ops.B2C_BF16, None, 1,
                                           torch.cuda.current_stream().cuda_stream)
        assert rc == 0, lib.b2c_last_error()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            call()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(reps):
            call()
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (5 * reps)
    nbytes = N * V * (2 + z.element_size()) + N * Vp * 2
    return {"us": ms * 1e3, "bytes": nbytes, "GB_per_s": nbytes / ms / 1e6}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--vocab", type=int, nargs="+", default=[5000, 4999])
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_teacher_dtype measures on a CUDA device"
    dev = torch.device("cuda:0")
    from imagecaptioner_b200 import _ops
    lib = _ops.load_library()
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        gpu, power = smi[0], float(smi[1])
    except Exception:           # nvidia-smi missing: the device name from torch, the power limit unknown
        gpu, power = torch.cuda.get_device_name(0), None
    out = {"gpu": gpu, "power_limit_w": power, "config": dict(bench.CFG, mode="eval, bf16 compute"), "results": {}}
    for V in args.vocab:
        cfg = dict(bench.CFG, V=V)
        built = {name: build(cfg, dev, dt) for name, dt in DTYPES.items()}
        times = {name: [] for name in DTYPES}
        loss = {}
        for name, (kd, _, _) in built.items():
            time_steps(kd, 5)
        for _ in range(args.rounds):
            for name, (kd, _, _) in built.items():
                ms, loss[name] = time_steps(kd, args.steps)
                times[name].append(ms)
        res = {}
        for name, (kd, pinned, resident) in built.items():
            res[name] = {"step_ms": min(times[name]), "step_ms_all": times[name], "loss": loss[name],
                         "token_pass": token_pass(lib, _ops, dev, V, cfg["B"] * cfg["T"], DTYPES[name]),
                         "e2e": e2e(kd, pinned, resident, args.steps)}
        out["results"][str(V)] = res
        del built
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
