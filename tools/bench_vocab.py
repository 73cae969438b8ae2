"""Vocabulary-size sweep of the graphed bf16 KD step at bench.py's configuration (B 512, T 20, E 256, H 512, L 2), one JSON line.

The reference's Vocabulary keeps every word above a frequency threshold, so V is rarely a multiple of 8; this measures what such a
V costs next to V = 5000:
  * step_ms[V]              graphed KD step (eval mode), CUDA events around `--steps` replays after `--warmup`
  * token_pass[V]           the token KD + CE pass alone at V = 5000 and 4999 (b2c_kd_token_loss_pitched for 4999 when the tree has it): time and
                            achieved bytes/s over its compulsory traffic (read y bf16 + z fp32, write dlogits bf16)
  * head_fwd_share          time of the tcgen05 GEMMs that write bf16 from K-major operands (the forward vocabulary head plus the
                            output_projection.0 contraction in front of it) next to the step's summed kernel time, per step at each V
                            (torch.profiler, separate pass)
  * validation              validate_student_model's per-batch body at V = 4999, logits materialised vs logits-free (when supported)
  * kernel_names[V]         the step's distinct kernel names (torch.profiler), for comparing two builds
  * gpu / power_limit_w     from the same process

--root DIR measures the tree at DIR (its package and its bench.py); B2C_LIB picks the library as usual.  Run two trees alternately
in one session to compare builds."""
import argparse
import json
import os
import subprocess
import sys

import torch


def token_pass(lib, _ops, dev, V, N):
    """b2c_kd_token_loss(_pitched) alone: time and achieved bytes/s over its compulsory traffic."""
    Vp = (V + 7) // 8 * 8
    g = torch.Generator(device=dev).manual_seed(0)
    y = torch.randn(N, V, generator=g, device=dev).bfloat16()
    z = torch.randn(N, V, generator=g, device=dev)
    t = torch.randint(1, V, (N,), generator=g, device=dev)
    nval = torch.full((1,), N, dtype=torch.int32, device=dev)
    rows = torch.empty(2, N, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    pitched = V % 8 != 0 and "b2c_kd_token_loss_pitched" in _ops.SYMBOLS
    dy = torch.empty(N, Vp if pitched else V, dtype=torch.bfloat16, device=dev)

    def call():
        if pitched:
            rc = lib.b2c_kd_token_loss_pitched(y.data_ptr(), z.data_ptr(), t.data_ptr(), N, V, 4.0, 0.7, 0.3, 1.0, nval.data_ptr(), dy.data_ptr(), Vp,
                                               rows[0].data_ptr(), rows[1].data_ptr(), _ops.B2C_BF16, st)
        else:
            rc = lib.b2c_kd_token_loss(y.data_ptr(), z.data_ptr(), t.data_ptr(), N, V, 4.0, 0.7, 0.3, 1.0, nval.data_ptr(), dy.data_ptr(),
                                       rows[0].data_ptr(), rows[1].data_ptr(), _ops.B2C_BF16, st)
        assert rc == 0, lib.b2c_last_error()
    for _ in range(5):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 50
    torch.cuda.synchronize(); e0.record()
    for _ in range(reps):
        call()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    nbytes = N * V * (2 + 4) + N * dy.shape[1] * 2
    return {"V": V, "rows": N, "pitched_entry": pitched, "us": ms * 1e3, "bytes": nbytes, "GB_per_s": nbytes / ms / 1e6,
            "note": "inputs ~307 MB > 126 MB L2, no flush between calls"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--vocab", default="5000,4999,5001")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args()
    root = os.path.abspath(args.root)
    sys.path.insert(0, root)
    import bench
    from imagecaptioner_b200 import _ops
    lib = _ops.load_library()
    assert torch.cuda.is_available(), "bench_vocab needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    out = {"root": root, "lib": _ops.LIB_PATH, "gpu": torch.cuda.get_device_name(dev), "power_limit_w": pl,
           "config": dict(bench.CFG, V=None), "steps": args.steps, "warmup": args.warmup,
           "step_ms": {}, "loss": {}, "kernel_names": {}, "head_fwd_share": {}}
    vocab = [int(v) for v in args.vocab.split(",")]
    for V in vocab:
        cfg = dict(bench.CFG, V=V)
        kd, *_ = bench.build_step(cfg, dev, 0, train_mode=False, single_process=True)
        ms, out5 = bench.time_steps(kd, args.steps, args.warmup, torch.cuda.synchronize, 1, dev)
        out["step_ms"][V], out["loss"][V] = ms, out5
        if not args.no_profile:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    kd.step()
                torch.cuda.synchronize()
            ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
            out["kernel_names"][V] = sorted({e.name for e in ev})
            total = sum(e.device_time for e in ev)
            head = sum(e.device_time for e in ev if "gemm_tc_kernel" in e.name and "__nv_bfloat16, 0>" in e.name and "false, false" in e.name)
            out["head_fwd_share"][V] = {"bf16_out_kmajor_gemm_us_per_step": head / 3, "all_kernels_us_per_step": total / 3}
        del kd
        torch.cuda.empty_cache()

    # token pass alone (N = T*B rows) at V = 5000 and 4999
    out["token_pass"] = {}
    for V in (5000, 4999):
        out["token_pass"][V] = token_pass(lib, _ops, dev, V, bench.CFG["T"] * bench.CFG["B"])

    # validation leg at V = 4999
    V = 4999
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from oracle import kd_oracle as O
    from tests.harness import build_student
    cfg = dict(bench.CFG, V=V)
    B, T, E, H, L = cfg["B"], cfg["T"], cfg["E"], cfg["H"], cfg["L"]
    model, projector = build_student(O.init_student_params(V, E, H, L, True, seed=0), O.init_projector_params(cfg["Et"], E, seed=1),
                                     V, E, H, L, True, cfg["Et"], dev)
    for m in (model.decoder, model.attention_refinement, projector):
        m.compute_dtype = torch.bfloat16
    batch = {k: (v.to(dev) if v is not None else None) for k, v in bench.make_batch(cfg, 99).items()}
    loss_mod = DistillationLoss(0.7, 0.2, 0.1, 4.0, vocab_size=V)
    val = {"supports_fused_validation": bool(model.supports_fused_validation())}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        t_out = {"logits": batch["teacher_logits"], "encoder_features": projector(batch["teacher_features"]), "hidden_states": None}

        def unfused():
            logits, enc, hids, _ = model(batch["encoder_features"], batch["captions_input"])
            return loss_mod.evaluate({"logits": logits, "encoder_features": enc, "hidden_states": hids}, t_out, batch["targets"])[1]

        def fused():
            return loss_mod.evaluate_fused(model, batch["encoder_features"], batch["captions_input"], t_out, batch["targets"])[1]
        legs = [("logits_materialised", unfused)] + ([("logits_free", fused)] if val["supports_fused_validation"] else [])
        for name, fn in legs:
            for _ in range(3):
                d = fn()
            torch.cuda.synchronize(); e0.record()
            for _ in range(10):
                d = fn()
            e1.record(); torch.cuda.synchronize()
            val[name] = {"ms_per_batch": e0.elapsed_time(e1) / 10, "total_loss": d["total_loss"]}
    out["validation_v4999"] = val
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
