"""Pin the oracle against the REAL reference and write the golden vectors.

Runs only where ``/root/reference`` exists (the build container).  It imports the
reference's own ``student_model`` / ``distillation_utils`` modules read-only, stubs the
ImageNet download in ``CNNEncoder`` (src/student_model.py:16) and swaps ``model.encoder``
for a pass-through so ``CaptioningStudent.forward`` runs unchanged on (B,49,E) features,
then:

  1. checks every oracle function against the reference module it restates, on seeded
     inputs (fp64 and fp32), and prints the max abs/rel error;
  2. writes ``tests/golden/*.pt``: inputs, parameters (reference state_dict), and the
     REFERENCE's outputs/loss/gradients, so that tests on a box without /root/reference
     (the GPU box) can still compare against the reference itself.

Usage:  PYTHONDONTWRITEBYTECODE=1 python oracle/pin_against_reference.py
"""
from __future__ import annotations

import os
import sys

os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")
sys.dont_write_bytecode = True

import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
REF_SRC = "/root/reference/src"

from oracle import kd_oracle as O  # noqa: E402
from tests.harness import save_golden  # noqa: E402


def load_reference():
    if not os.path.isdir(REF_SRC):
        raise SystemExit("reference not present; the golden vectors in tests/golden are the pin")
    sys.path.insert(0, REF_SRC)
    import torchvision
    import student_model as ref_sm            # noqa
    import distillation_utils as ref_du       # noqa
    ref_sm.models.resnet50 = lambda weights=None: torchvision.models.resnet50(weights=None)
    return ref_sm, ref_du


class _PassThrough(nn.Module):
    def __init__(self):
        super().__init__()
        self.adaptive_pool = nn.AdaptiveAvgPool2d((7, 7))

    def forward(self, x):
        return x.reshape(-1, 49, x.shape[-1])      # (49,E) from caption_image -> (1,49,E)


def build_reference_student(ref_sm, V, E, H, L, seed, refinement=True, logit_scale=1.0):
    torch.manual_seed(seed)
    dec = ref_sm.LSTMDecoder(V, E, H, L, dropout=0.0)
    model = ref_sm.CaptioningStudent.__new__(ref_sm.CaptioningStudent)
    nn.Module.__init__(model)
    model.vocab_size, model.embed_size, model.hidden_size = V, E, H
    model.encoder = _PassThrough()
    model.use_attention_refinement = refinement
    if refinement:
        model.attention_refinement = ref_sm.AttentionRefinement(embed_size=E)
    model.decoder = dec
    with torch.no_grad():
        model.decoder.output_projection[3].weight.mul_(logit_scale)
        # non-zero LSTM biases so the bias path is exercised (reference init is zero)
        for n, p_ in model.decoder.lstm.named_parameters():
            if "bias" in n:
                p_.uniform_(-0.05, 0.05)
    model.eval()
    return model


def ref_kd_step(ref_du, model, projector, batch, alpha, beta, gamma, temperature, V):
    model.zero_grad(set_to_none=True)
    projector.zero_grad(set_to_none=True)
    feats = batch["encoder_features"].clone().requires_grad_(True)
    outputs, enc, hids, atts = model(feats, batch["captions_input"])
    t_out = {"logits": batch["teacher_logits"],
             "encoder_features": projector(batch["teacher_features"]),
             "hidden_states": None if batch["teacher_hiddens"] is None
             else [batch["teacher_hiddens"][t] for t in range(batch["teacher_hiddens"].shape[0])]}
    s_out = {"logits": outputs, "encoder_features": enc, "hidden_states": hids}
    loss_mod = ref_du.DistillationLoss(alpha, beta, gamma, temperature, vocab_size=V)
    total, loss_dict = loss_mod(s_out, t_out, batch["targets"])
    total.backward()
    return {
        "loss": loss_dict,
        "grads": {k: v.grad.detach().clone() for k, v in model.named_parameters() if v.grad is not None},
        "proj_grads": {k: v.grad.detach().clone() for k, v in projector.named_parameters() if v.grad is not None},
        "d_encoder_features": feats.grad.detach().clone(),
        "logits": outputs.detach().clone(),
        "hidden_states": torch.stack([h.detach() for h in hids]),
        "attention_weights": torch.stack([a.detach() for a in atts]),
        "teacher_projected": t_out["encoder_features"].detach().clone(),
    }


def relerr(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def compare(tag, got, ref, tol):
    worst = 0.0
    for k in ("logits", "hidden_states", "attention_weights", "teacher_projected", "d_encoder_features"):
        worst = max(worst, relerr(got[k], ref[k]))
    for k, v in ref["grads"].items():
        worst = max(worst, relerr(got["grads"][k], v))
    for k, v in ref["proj_grads"].items():
        worst = max(worst, relerr(got["proj_grads"][k], v))
    for k, v in ref["loss"].items():
        worst = max(worst, abs(got["loss"][k] - v) / (abs(v) + 1e-30))
    status = "OK " if worst < tol else "FAIL"
    print(f"[{status}] {tag}: worst rel err oracle-vs-reference = {worst:.3e} (tol {tol:g})")
    return worst < tol


ET_SMALL = 40   # teacher feature width of the small fixtures (197 tokens kept: the 197->49 pooling rule is the point)

CASES = {
    # name: (B, T, V, E, H, L, refinement, alpha, beta, gamma, temperature, teacher_hiddens)
    "kd_small_default": (4, 6, 104, 32, 64, 2, True, 0.7, 0.2, 0.1, 4.0, True),
    "kd_small_large_variant": (3, 5, 203, 48, 96, 3, True, 0.5, 0.2, 0.1, 4.0, True),
    "kd_small_ce_heavy_nohid": (5, 7, 57, 32, 64, 2, False, 0.3, 0.1, 0.0, 2.0, False),
}


def main():
    ref_sm, ref_du = load_reference()
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    ok = True
    for name, (B, T, V, E, H, L, refine, a, b, g, temp, th) in CASES.items():
        for dtype, tol in ((torch.float64, 1e-9), (torch.float32, 2e-4)):
            torch.set_default_dtype(dtype)
            model = build_reference_student(ref_sm, V, E, H, L, seed=7, refinement=refine)
            torch.manual_seed(11)
            projector = ref_du.FeatureProjector(ET_SMALL, E, 197, 49).eval()
            batch = O.synthetic_batch(B, T, V, E, H, Et=ET_SMALL, seed=99, teacher_hiddens=th)
            batch = {k: (v.to(dtype) if (v is not None and v.is_floating_point()) else v) for k, v in batch.items()}
            ref = ref_kd_step(ref_du, model, projector, batch, a, b, g, temp, V)
            params = {k: v.detach().clone() for k, v in model.state_dict().items()
                      if not k.startswith("encoder.")}
            pparams = {k: v.detach().clone() for k, v in projector.state_dict().items()}
            got = O.kd_step(params, pparams, batch, a, b, g, temp, use_refinement=refine, dtype=dtype)
            ok &= compare(f"{name}/{str(dtype)[6:]}", got, ref, tol)
            if dtype == torch.float32:
                save_golden({"meta": dict(B=B, T=T, V=V, E=E, H=H, L=L, refinement=refine, alpha=a, beta=b,
                                          gamma=g, temperature=temp, torch=torch.__version__,
                                          generator="oracle/pin_against_reference.py (reference modules, fp32 CPU)"),
                             "params": params, "proj_params": pparams, "batch": batch, "reference": ref}, name)
        torch.set_default_dtype(torch.float32)

    # ---- greedy decode: reference step methods in a batched loop + caption_image at B=1 ----
    B, V, E, H, L, max_len = 6, 120, 32, 64, 2, 12
    model = build_reference_student(ref_sm, V, E, H, L, seed=21, refinement=True, logit_scale=8.0)
    params = {k: v.detach().clone() for k, v in model.state_dict().items() if not k.startswith("encoder.")}
    feats = torch.randn(B, 49, E, generator=torch.Generator().manual_seed(5))

    class Vocab:                                  # the slice of data_loader.Vocabulary caption_image touches
        def __init__(self, n):
            self.itos = {0: "<PAD>", 1: "<START>", 2: "<END>", 3: "<UNK>"}
            self.itos.update({i: f"w{i}" for i in range(4, n)})
            self.stoi = {v: k for k, v in self.itos.items()}

    vocab = Vocab(V)
    with torch.no_grad():
        refined = model.attention_refinement(feats)
        toks, lengths, margins = O.greedy_decode(params, refined, max_len)
        ref_caps = [model.caption_image(feats[i], vocab, max_length=max_len) for i in range(B)]
    for i in range(B):
        words = [vocab.itos[int(t)] for t in toks[: int(lengths[i]), i]]
        if words != ref_caps[i]:
            ok = False
            print(f"[FAIL] greedy sample {i}: oracle {words} vs caption_image {ref_caps[i]}")
    print(f"[{'OK ' if ok else 'FAIL'}] greedy decode: {B} captions identical to caption_image; "
          f"min top1-top2 margin {float(margins.min()):.3e}; lengths {lengths.tolist()}")
    torch.save({"meta": dict(B=B, V=V, E=E, H=H, L=L, max_len=max_len, torch=torch.__version__),
                "params": params, "features": feats, "refined": refined,
                "reference": {"captions": ref_caps, "tokens": toks, "lengths": lengths, "min_margin": float(margins.min())}},
               os.path.join(ROOT, "tests", "golden", "greedy_small.pt"))

    # ---- the one value-free pin the reference's own test holds: FeatureProjector shape ----
    fp = ref_du.FeatureProjector(384, 256, 197, 64).eval()         # test_dimension_fix.py:16-43
    x = torch.randn(2, 197, 384)
    mine = O.feature_projector({k: v for k, v in fp.state_dict().items()}, x, 64)
    assert tuple(mine.shape) == (2, 64, 256) and relerr(mine, fp(x).detach()) < 1e-5
    print("[OK ] FeatureProjector(384,256,197,64) -> (2,64,256), values match")

    # ---- config-1 shape summary (full tensors are too big to commit; keep scalars + samples) ----
    B, T, V, E, H, L = 16, 20, 5000, 256, 512, 2
    model = build_reference_student(ref_sm, V, E, H, L, seed=3, refinement=True)
    torch.manual_seed(4)
    projector = ref_du.FeatureProjector(384, E, 197, 49).eval()
    # parameters come from the oracle's seeded initialiser so the GPU box can rebuild them
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(384, E, seed=1)
    model.load_state_dict({**params}, strict=False)
    projector.load_state_dict(pparams)
    batch = O.synthetic_batch(B, T, V, E, H, seed=1234)
    ref = ref_kd_step(ref_du, model, projector, batch, 0.7, 0.2, 0.1, 4.0, V)
    got = O.kd_step(params, pparams, batch)
    ok &= compare("config1 (B16 T20 V5000)/float32", got, ref, 2e-4)
    summary = {"meta": dict(B=B, T=T, V=V, E=E, H=H, L=L, param_seed=0, proj_seed=1, batch_seed=1234,
                            torch=torch.__version__),
               "loss": ref["loss"],
               "grad_norms": {k: float(v.norm()) for k, v in ref["grads"].items()},
               "proj_grad_norms": {k: float(v.norm()) for k, v in ref["proj_grads"].items()},
               "d_encoder_features_norm": float(ref["d_encoder_features"].norm()),
               "logits_sample": ref["logits"][::5, ::4, ::499].clone(),
               "logits_norm": float(ref["logits"].norm())}
    torch.save(summary, os.path.join(ROOT, "tests", "golden", "config1_summary.pt"))
    print("ALL PINNED" if ok else "PIN FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
