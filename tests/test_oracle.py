"""CPU: the oracle against the committed golden vectors (generated from the REAL reference modules by
oracle/pin_against_reference.py) and the hand-derived backward blueprint against autograd."""
import os

import pytest
import torch

from oracle import kd_oracle as O
from oracle import manual_backward as M
from tests.harness import GOLDEN, load_golden, relerr

KD_CASES = ["kd_small_default", "kd_small_large_variant", "kd_small_ce_heavy_nohid"]


@pytest.mark.parametrize("name", KD_CASES)
def test_oracle_matches_reference_golden(name):
    g = load_golden(name)
    m, ref = g["meta"], g["reference"]
    got = O.kd_step(g["params"], g["proj_params"], g["batch"], m["alpha"], m["beta"], m["gamma"], m["temperature"],
                    use_refinement=m["refinement"])
    tol = 2e-4   # fp32 CPU vs fp32 CPU, different op order
    for k in ("logits", "hidden_states", "attention_weights", "teacher_projected", "d_encoder_features"):
        assert relerr(got[k], ref[k]) < tol, k
    for k, v in ref["grads"].items():
        assert relerr(got["grads"][k], v) < tol, k
    for k, v in ref["proj_grads"].items():
        assert relerr(got["proj_grads"][k], v) < tol, k
    for k, v in ref["loss"].items():
        assert abs(got["loss"][k] - v) <= tol * max(abs(v), 1e-6), k


def test_oracle_greedy_matches_caption_image_golden():
    g = torch.load(os.path.join(GOLDEN, "greedy_small.pt"), weights_only=False)
    toks, lengths, margins = O.greedy_decode(g["params"], g["refined"], g["meta"]["max_len"])
    assert torch.equal(toks, g["reference"]["tokens"]) and torch.equal(lengths, g["reference"]["lengths"])
    itos = {0: "<PAD>", 1: "<START>", 2: "<END>", 3: "<UNK>"}
    for b, words in enumerate(g["reference"]["captions"]):        # caption_image's own output, word by word
        mine = [itos.get(int(t), f"w{int(t)}") for t in toks[: int(lengths[b]), b]]
        assert mine == words
    assert float(margins.min()) > 1e-3, "fixture is ill-conditioned for token-id parity"


def test_oracle_config1_summary():
    g = torch.load(os.path.join(GOLDEN, "config1_summary.pt"), weights_only=False)
    m = g["meta"]
    params = O.init_student_params(m["V"], m["E"], m["H"], m["L"], True, seed=m["param_seed"])
    pparams = O.init_projector_params(384, m["E"], seed=m["proj_seed"])
    batch = O.synthetic_batch(m["B"], m["T"], m["V"], m["E"], m["H"], seed=m["batch_seed"])
    got = O.kd_step(params, pparams, batch)
    for k, v in g["loss"].items():
        assert abs(got["loss"][k] - v) <= 2e-4 * max(abs(v), 1e-6), k
    assert relerr(got["logits"][::5, ::4, ::499], g["logits_sample"]) < 2e-4
    for k, v in g["grad_norms"].items():
        assert abs(float(got["grads"][k].norm()) - v) <= 1e-3 * max(v, 1e-9), k


def test_feature_projector_shape_pin():
    """The one pin the reference's own test holds (test_dimension_fix.py:16-43): (2,197,384) -> (2,64,256)."""
    p = O.init_projector_params(384, 256, seed=3)
    out = O.feature_projector(p, torch.randn(2, 197, 384), 64)
    assert tuple(out.shape) == (2, 64, 256)


def test_adaptive_pool_rule():
    x = torch.randn(2, 197, 8)
    ref = torch.nn.functional.adaptive_avg_pool1d(x.transpose(1, 2), 49).transpose(1, 2)
    assert relerr(O.adaptive_avg_pool_tokens(x, 49), ref) < 1e-6


@pytest.mark.parametrize("dims", [(4, 6, 104, 32, 64, 2), (3, 5, 203, 48, 96, 3), (2, 1, 57, 16, 24, 1)])
def test_manual_backward_blueprint_matches_autograd(dims):
    B, T, V, E, H, L = dims
    torch.manual_seed(0)
    p = {k: v.double() for k, v in O.init_student_params(V, E, H, L, False, seed=3).items()}
    for k in p:
        if "bias" in k:
            p[k] = torch.randn_like(p[k]) * 0.05
    b = O.synthetic_batch(B, T, V, E, H, seed=5)
    feats, caps = b["encoder_features"].double(), b["captions_input"]
    P = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    f = feats.clone().requires_grad_(True)
    out, hids, atts = O.decoder_forward(P, f, caps)
    dlog, dh = torch.randn_like(out), torch.randn(T, B, H, dtype=torch.float64)
    ((out * dlog).sum() + sum((hids[t] * dh[t]).sum() for t in range(T))).backward()
    lg, hid, w, sv = M.decoder_forward_saved(p, feats, caps)
    assert relerr(lg, out.detach()) < 1e-12 and relerr(w, torch.stack(atts).detach()) < 1e-12
    G, dF = M.decoder_backward_manual(p, feats, caps, sv, dlog, dh)
    assert relerr(dF, f.grad) < 1e-10
    for k in P:
        assert relerr(G[k], P[k].grad) < 1e-10, k


@pytest.mark.parametrize("dims", [(4, 6, 104, 32, 64, 2), (3, 5, 203, 48, 96, 3), (2, 3, 57, 16, 24, 1)])
def test_manual_backward_v2_fold_matches_autograd(dims):
    """v2 dataflow (attention_combine folded into layer 0's gate contraction — what csrc/api.cu runs) vs autograd."""
    B, T, V, E, H, L = dims
    p = {k: v.double() for k, v in O.init_student_params(V, E, H, L, False, seed=3).items()}
    gen = torch.Generator().manual_seed(1)
    for k in p:
        if "bias" in k:
            p[k] = torch.randn(p[k].shape, generator=gen, dtype=torch.float64) * 0.05
    b = O.synthetic_batch(B, T, V, E, H, seed=5)
    feats, caps = b["encoder_features"].double(), b["captions_input"]
    P = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    f = feats.clone().requires_grad_(True)
    out, hids, atts = O.decoder_forward(P, f, caps)
    dlog, dh = torch.randn(out.shape, generator=gen, dtype=torch.float64), torch.randn(T, B, H, generator=gen, dtype=torch.float64)
    ((out * dlog).sum() + sum((hids[t] * dh[t]).sum() for t in range(T))).backward()
    lg, hid, w, sv = M.decoder_forward_saved_v2(p, feats, caps)
    assert relerr(lg, out.detach()) < 1e-12 and relerr(w, torch.stack(atts).detach()) < 1e-12
    G, dF = M.decoder_backward_manual_v2(p, feats, caps, sv, dlog, dh)
    assert relerr(dF, f.grad) < 1e-10
    for k in P:
        assert relerr(G[k], P[k].grad) < 1e-10, k


def test_closed_form_token_gradient():
    torch.manual_seed(1)
    y = torch.randn(5, 3, 50, dtype=torch.float64, requires_grad=True)
    z = torch.randn(5, 3, 50, dtype=torch.float64) * 2
    t = torch.randint(0, 50, (5, 3)); t[0, 0] = 0
    (0.7 * O.token_kd(y, z, 4.0) + 0.3 * O.cross_entropy_ignore_pad(y, t)).backward()
    assert relerr(M.kd_token_grad(y.detach(), z, t, 4.0, 0.7, 0.3), y.grad) < 1e-12


def test_loss_edge_cases():
    # teacher hiddens None -> hidden term is exactly 0 (what TeacherWrapper always produces, distillation_utils.py:291)
    assert float(O.hidden_kd(None, [torch.zeros(2, 4)])) == 0.0
    # cosine eps semantics measured on the reference (SURVEY.md §8c): two zero vectors -> 1.0
    z = [torch.zeros(3, 8)]
    assert abs(float(O.hidden_kd(z, z)) - 0.3) < 1e-7
    with pytest.raises(ValueError):
        O.feature_kd(torch.zeros(2, 49, 8), torch.zeros(2, 49, 16))
    # list truncation to the shorter side
    s = [torch.randn(2, 8) for _ in range(5)]
    assert abs(float(O.hidden_kd(s, s[:3])) - float(O.hidden_kd(s[:3], s[:3]))) < 1e-7


def test_validation_oracle_matches_reference_fixture():
    """oracle bleu1 / eval_step vs tests/golden/validation_case.pt (written by oracle/pin_validation.py from the reference's
    compute_bleu_score and logits.argmax)."""
    import os
    from tests.harness import GOLDEN
    fx = torch.load(os.path.join(GOLDEN, "validation_case.pt"), weights_only=False)
    got = O.bleu1(fx["bleu"]["pred"], fx["bleu"]["targets"])
    assert torch.allclose(got, fx["bleu"]["reference"], atol=1e-6)
    assert float(got[0]) == 0.0 and abs(float(got[1]) - 1.0) < 1e-6        # empty target set; {5} vs {5, 9}
    case = torch.load(os.path.join(GOLDEN, "kd_small_default.pt"), weights_only=False)
    ev = O.eval_step(case["params"], case["proj_params"], case["batch"])
    assert torch.equal(ev["predicted_tokens"], fx["kd_small_default"]["predicted_tokens"])
    assert torch.allclose(ev["bleu"], fx["kd_small_default"]["bleu"], atol=1e-6)


@pytest.mark.parametrize("case", ["default", "identity_projection_3_layers_no_hiddens"])
def test_stock_module_restatement_matches_oracle(case):
    """oracle/eager_torch.py (the reference's composition of stock torch.nn modules: nn.LSTM stepped per token, nn.MultiheadAttention,
    F.kl_div, ...) against the plain-arithmetic oracle that is pinned on the real reference: every output, loss part and gradient.
    It is the GPU-side baseline of bench.py and the yardstick of the bf16 tolerance (tests/harness.py:autocast_reference_errors)."""
    from oracle import eager_torch as ET
    from tests.harness import step_errors
    if case == "default":
        V, E, H, L, B, T, Et, refine, hid = 120, 32, 64, 2, 6, 5, 24, True, True
    else:
        V, E, H, L, B, T, Et, refine, hid = 60, 32, 48, 3, 4, 3, 32, False, False
    params = O.init_student_params(V, E, H, L, refine, seed=3)
    pparams = O.init_projector_params(Et, E, seed=4)
    batch = O.synthetic_batch(B, T, V, E, H, Et=Et, seed=5, teacher_hiddens=hid)
    ref = O.kd_step(params, pparams, batch, use_refinement=refine)
    model, proj = ET.build(params, pparams, V, E, H, L, refine, Et)
    got = ET.kd_step(model, proj, batch)
    errs = step_errors(got, ref, metric="max")
    assert max(errs.values()) < 2e-5, sorted(errs.items(), key=lambda kv: -kv[1])[:3]
    # the autocast form runs on the CPU too (bf16): a finite, small but non-zero deviation
    errs16 = step_errors(ET.kd_step(model, proj, batch, torch.bfloat16), ref, metric="l2")
    assert 1e-4 < max(errs16.values()) < 0.5


def test_oracle_decoder_forward_with_initial_hidden_state_matches_reference_fixture():
    """oracle.decoder_forward(..., hidden=(h0, c0)) against the reference's own LSTMDecoder.forward(hidden=...) outputs
    (tests/golden/hidden_init_case.pt, written by oracle/pin_hidden.py from the real reference module)."""
    import os
    g = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hidden_init_case.pt"), weights_only=False)
    out, hids, atts = O.decoder_forward(g["params"], g["feats"], g["captions"], hidden=(g["h0"], g["c0"]))
    ref = g["reference"]
    assert float((out - ref["outputs"]).abs().max()) < 2e-5
    assert float((torch.stack(hids) - ref["hidden_states"]).abs().max()) < 2e-5
    assert float((torch.stack(atts) - ref["attention_weights"]).abs().max()) < 2e-5
    # and the zero state is the default
    z = torch.zeros_like(g["h0"])
    a = O.decoder_forward(g["params"], g["feats"], g["captions"])[0]
    b = O.decoder_forward(g["params"], g["feats"], g["captions"], hidden=(z, z))[0]
    assert torch.equal(a, b)
