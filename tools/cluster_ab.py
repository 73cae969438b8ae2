"""A/B check of a process-level switch of the native path: the same bf16 KD step is run in two subprocesses (VAR=on / VAR=off; the
switches are read once per process), every output and gradient is compared, and the decoder forward is timed.  Default: the cluster
recurrence kernel (csrc/recur_cluster.cuh, B2C_CLUSTER=1 / 0) against the per-step kernels.
Usage: python tools/cluster_ab.py [--env VAR=on,off] [--tol 2e-2] [B ...]        (default: B2C_CLUSTER=1,0; sizes 16 35 512)"""
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(B, out):
    import torch
    from oracle import kd_oracle as O
    from tests.harness import build_student, run_kd_step
    dev = torch.device("cuda:0")
    T, V, E, H, L = 20, 5000, 256, 512, 2
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(384, E, seed=1)
    batch = O.synthetic_batch(B, T, V, E, H, Et=384, seed=7)
    model, projector = build_student(params, pparams, V, E, H, L, True, 384, dev)
    got = run_kd_step(model, projector, batch, dev, torch.bfloat16)
    torch.cuda.synchronize()
    # forward-only timing of the decoder (eager launches: host-bound for the per-step path, one launch for the cluster path)
    feats = batch["encoder_features"].to(dev)
    cap = batch["captions_input"].to(dev)
    model.decoder.compute_dtype = torch.bfloat16
    with torch.no_grad():
        for _ in range(3):
            model.decoder(feats, cap)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(10):
            model.decoder(feats, cap)
        torch.cuda.synchronize()
        got["fwd_ms"] = (time.perf_counter() - t0) * 100.0
    torch.save(got, out)


def main():
    import torch
    from tests.harness import relerr, relerr_l2
    argv = sys.argv[1:]
    var, on, off, tol = "B2C_CLUSTER", "1", "0", 2e-2
    while argv and argv[0].startswith("--"):
        if argv[0] == "--env":
            var, vals = argv[1].split("=")
            on, off = vals.split(",")
        elif argv[0] == "--tol":
            tol = float(argv[1])
        argv = argv[2:]
    sizes = [int(a) for a in argv] or [16, 35, 512]
    tmp = tempfile.mkdtemp(prefix="cluster_ab_")
    ok = True
    for B in sizes:
        res = {}
        for mode in (on, off):
            out = os.path.join(tmp, f"ab_{var}_{B}_{mode}.pt")
            env = dict(os.environ)
            env[var] = mode
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", str(B), out], env=env, capture_output=True, text=True, timeout=600)
            if r.returncode != 0:
                print(f"B={B} {var}={mode}: child failed\n{r.stdout[-2000:]}\n{r.stderr[-3000:]}")
                ok = False
                break
            res[mode] = torch.load(out, weights_only=False)
            os.remove(out)
        if len(res) < 2:
            continue
        a, b = res[on], res[off]
        rows = [(k, relerr(a[k], b[k]), relerr_l2(a[k], b[k])) for k in ("logits", "hidden_states", "attention_weights", "d_encoder_features")]
        rows += [("grad:" + k, relerr(a["grads"][k], v), relerr_l2(a["grads"][k], v)) for k, v in b["grads"].items()]
        worst = max(rows, key=lambda r: r[2])
        print(f"B={B}: loss {var}={on} {a['loss']['total_loss']:.6f} / {var}={off} {b['loss']['total_loss']:.6f}; decoder forward {a['fwd_ms']:.3f} ms vs {b['fwd_ms']:.3f} ms (eager launches)")
        for k, e, e2 in rows[:4]:
            print(f"   {k:28s} max-norm {e:.3e}  L2 {e2:.3e}")
        print(f"   worst gradient: {worst[0]} L2 {worst[2]:.3e}")
        bad = [r for r in rows if not (r[2] < tol)]
        if bad:
            ok = False
            print("   MISMATCH:", bad[:6])
    shutil.rmtree(tmp, ignore_errors=True)
    print("cluster A/B:" if var == "B2C_CLUSTER" else f"{var} A/B:", "OK" if ok else "FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        child(int(sys.argv[2]), sys.argv[3])
    else:
        sys.exit(main())
