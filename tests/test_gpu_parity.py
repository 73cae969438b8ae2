"""GPU: the whole KD step and greedy decode through the public modules against the golden vectors produced by the
REAL reference (tests/golden, generator oracle/pin_against_reference.py) and against the oracle at larger sizes."""
import os

import pytest
import torch

from oracle import kd_oracle as O
from tests.harness import (GOLDEN, autocast_reference_errors, build_student, compare_step, compare_step_calibrated, load_golden, relerr, relerr_l2,
                           run_kd_step, step_errors, to_device)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FP32_TOL = 1e-4      # BASELINE.json north_star: loss and gradients within 1e-4 relative in fp32
BF16_TOL = 2e-2      # ... and 2e-2 in bf16
KD_CASES = ["kd_small_default", "kd_small_large_variant", "kd_small_ce_heavy_nohid"]
# gradients of the Linear layers that sit directly behind a ReLU: in bf16 mode a few mask elements flip (DESIGN.md section 2)
GATED = ("grad:decoder.output_projection.0.weight", "grad:decoder.output_projection.0.bias",
         "grad:attention_refinement.ffn.0.weight", "grad:attention_refinement.ffn.0.bias",
         "pgrad:feature_projection.0.weight", "pgrad:feature_projection.0.bias")


def _golden_step(name, dtype):
    g = load_golden(name)
    m = g["meta"]
    Et = g["batch"]["teacher_features"].shape[-1]
    model, projector = build_student(g["params"], g["proj_params"], m["V"], m["E"], m["H"], m["L"], m["refinement"], Et, DEV)
    got = run_kd_step(model, projector, g["batch"], DEV, dtype, m["alpha"], m["beta"], m["gamma"], m["temperature"])
    return got, g["reference"]


@pytest.mark.parametrize("name", KD_CASES)
def test_kd_step_fp32_matches_reference(name):
    got, ref = _golden_step(name, torch.float32)
    compare_step(got, ref, FP32_TOL)


@pytest.mark.parametrize("name", KD_CASES)
def test_kd_step_bf16_matches_reference(name):
    """bf16 mode against the reference's fp32 golden vectors: every tensor within max(2e-2, 1.2 x the error the REFERENCE's own
    arithmetic shows under torch.autocast(bf16) on the same inputs) -- no hand-set per-tensor factors."""
    got, ref = _golden_step(name, torch.bfloat16)
    g = load_golden(name)
    ref_err = autocast_reference_errors(g["params"], g["proj_params"], g["meta"], g["batch"], ref, DEV, use_refinement=g["meta"]["refinement"])
    compare_step_calibrated(got, ref, ref_err, BF16_TOL)


def _config1():
    g = torch.load(os.path.join(GOLDEN, "config1_summary.pt"), weights_only=False)
    m = g["meta"]
    params = O.init_student_params(m["V"], m["E"], m["H"], m["L"], True, seed=m["param_seed"])
    pparams = O.init_projector_params(384, m["E"], seed=m["proj_seed"])
    batch = O.synthetic_batch(m["B"], m["T"], m["V"], m["E"], m["H"], seed=m["batch_seed"])
    return g, m, params, pparams, batch


def test_config1_fp32_against_reference_summary_and_oracle():
    """BASELINE config 1 (B16 T20 V5000 E256 H512 L2): loss + gradient norms pinned by the reference, full tensors by the oracle."""
    g, m, params, pparams, batch = _config1()
    model, projector = build_student(params, pparams, m["V"], m["E"], m["H"], m["L"], True, 384, DEV)
    got = run_kd_step(model, projector, batch, DEV, torch.float32)
    for k, v in g["loss"].items():
        assert abs(got["loss"][k] - v) <= FP32_TOL * max(abs(v), 1e-6), (k, got["loss"][k], v)
    for k, v in g["grad_norms"].items():
        assert abs(float(got["grads"][k].norm()) - v) <= 5e-4 * max(v, 1e-9), k
    assert relerr(got["logits"][::5, ::4, ::499], g["logits_sample"]) < FP32_TOL
    ref = O.kd_step(params, pparams, batch)
    compare_step(got, ref, 2e-4)       # oracle itself is fp32-CPU (7e-5 from the reference at this size)


def test_config1_bf16_within_north_star_tolerance():
    """bf16 mode vs the fp32 oracle at config-1 shapes: 2e-2 relative, per tensor in the L2 norm.
    The two output_projection.0 gradients sit behind the ReLU: at the reference's initialisation its pre-activations
    are concentrated near 0 (|b1| <= 0.044, h ~ 0), so a ~0.3 % forward difference flips the mask of ~0.1 % of the
    elements and each flip moves the gradient by a whole term (measured: oracle-side simulation in DESIGN.md, 'bf16
    parity').  Those two are held to 4x the tolerance; everything else, and the loss, to 2e-2."""
    g, m, params, pparams, batch = _config1()
    model, projector = build_student(params, pparams, m["V"], m["E"], m["H"], m["L"], True, 384, DEV)
    got = run_kd_step(model, projector, batch, DEV, torch.bfloat16)
    ref = O.kd_step(to_device(params, DEV), to_device(pparams, DEV), to_device(batch, DEV), dtype=torch.float64)     # fp64 oracle (on the GPU: speed only)
    # The yardstick: the reference's own stock-module arithmetic under torch.autocast(bf16) on the same inputs.  Every tensor of the
    # native bf16 mode must be within max(2e-2, 1.2 x that error); the measured pairs are printed (and tabulated in DESIGN.md section 2).
    ref_err = autocast_reference_errors(params, pparams, m, batch, ref, DEV)
    compare_step_calibrated(got, ref, ref_err, BF16_TOL)


def test_greedy_decode_token_ids_identical_fp32():
    g = torch.load(os.path.join(GOLDEN, "greedy_small.pt"), weights_only=False)
    m = g["meta"]
    model, _ = build_student(g["params"], {}, m["V"], m["E"], m["H"], m["L"], True, m["E"], DEV)
    toks, lengths = model.decoder.greedy(g["refined"].to(DEV), m["max_len"])
    assert torch.equal(toks.cpu(), g["reference"]["tokens"])
    assert torch.equal(lengths.cpu().long(), g["reference"]["lengths"])

    class Vocab:
        itos = {0: "<PAD>", 1: "<START>", 2: "<END>", 3: "<UNK>", **{i: f"w{i}" for i in range(4, m["V"])}}
        stoi = {v: k for k, v in itos.items()}
    # caption_image (refinement included) reproduces the reference's own captions word for word
    for b in range(m["B"]):
        assert model.caption_image(g["features"][b].to(DEV), Vocab, max_length=m["max_len"]) == g["reference"]["captions"][b]
    assert not model.training                                   # caption_image leaves the model in eval() like the reference


def test_greedy_decode_with_end_tokens_against_oracle():
    """Bias the <END> logit so captions end at different steps; lengths and the tokens before <END> must match."""
    V, E, H, L, B, max_len = 60, 32, 64, 2, 16, 10
    params = O.init_student_params(V, E, H, L, False, seed=9, logit_scale=10.0)
    params["decoder.output_projection.3.bias"][2] += 1.2
    feats = torch.randn(B, 49, E, generator=torch.Generator().manual_seed(2))
    toks, lengths, margins = O.greedy_decode(params, feats, max_len)
    assert float(margins.min()) > 1e-3 and 0 < int((lengths < max_len).sum()) <= B
    model, _ = build_student(params, {}, V, E, H, L, False, E, DEV)
    t2, l2 = model.decoder.greedy(feats.to(DEV), max_len)
    assert torch.equal(l2.cpu().long(), lengths) and torch.equal(t2.cpu(), toks)


def test_training_mode_dropout_is_consistent():
    """Dropout on: forward is reproducible for a fixed seed, the keep rate is ~1-p and backward uses the same mask
    (finite-difference check of one directional derivative in fp32)."""
    from imagecaptioner_b200 import _ops
    V, E, H, L, B, T = 80, 32, 64, 2, 6, 5
    params = O.init_student_params(V, E, H, L, False, seed=4)
    model, _ = build_student(params, {}, V, E, H, L, False, E, DEV, dropout=0.3)
    dec = model.decoder
    plist = dec._param_list()
    feats = torch.randn(B, 49, E, device=DEV)
    cap = torch.randint(1, V, (T, B), device=DEV)

    counter = torch.zeros(1, dtype=torch.int64, device=DEV)
    opts = _ops.CallOptions(seed_dev=counter)

    def fwd(f, seed=123):
        return _ops.DecoderFunction.apply(f, cap, torch.float32, 0.3, seed, L, None, opts, None, *plist)
    y1, h1, _ = fwd(feats); y2, _, _ = fwd(feats); y3, _, _ = fwd(feats, seed=124)
    assert torch.equal(y1, y2) and not torch.equal(y1, y3)
    # the device-side step counter (B2CDropout.seed_dev) changes the mask without touching the by-value seed: a CUDA graph, whose
    # kernel arguments are frozen at capture, draws a fresh mask on every replay once the counter is bumped inside the graph
    _ops.bump_counter(counter)
    y4, _, _ = fwd(feats)
    assert int(counter.item()) == 1 and not torch.equal(y1, y4)
    counter.zero_()
    assert torch.equal(fwd(feats)[0], y1)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fwd(feats)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(graph):
        _ops.bump_counter(counter)
        yg = fwd(feats)[0]
    graph.replay(); torch.cuda.synchronize(); r1 = yg.clone()
    graph.replay(); torch.cuda.synchronize(); r2 = yg.clone()
    assert int(counter.item()) == 2 and not torch.equal(r1, r2)          # two replays, two different masks
    assert torch.equal(r1, y4)                                           # replay 1 saw counter == 1, like the eager call above
    counter.zero_()
    f = feats.clone().requires_grad_(True)
    y, _, _ = fwd(f)
    w = torch.randn_like(y)
    (y * w).sum().backward()
    # a backward that regenerated a DIFFERENT mask would be off by O(p) = 30 %; ReLU kinks and fp32 round-off limit the
    # finite difference itself to a few per cent, so average three directions and allow 6 %
    eps, errs = 5e-3, []
    for i in range(3):
        d = torch.randn(feats.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(100 + i))
        num = (((fwd(feats + eps * d)[0].double() - fwd(feats - eps * d)[0].double()) * w.double()).sum() / (2 * eps)).item()
        ana = (f.grad.double() * d.double()).sum().item()
        scale = float(f.grad.double().norm() * d.double().norm()) / (d.numel() ** 0.5)     # typical |<grad, d>| for a random direction
        errs.append(abs(num - ana) / scale)
    assert sum(errs) / len(errs) < 6e-2, errs


def test_data_parallel_normaliser_matches_global_batch():
    """Two half-batches with the GLOBAL non-PAD count and ce_mult = 2, averaged like the gradient all-reduce does,
    reproduce the full-batch gradient (SURVEY.md §8e exactness caveat), here emulated on one GPU through the C ABI."""
    from imagecaptioner_b200 import _ops
    lib = _ops.load_library()
    g = torch.Generator().manual_seed(5)
    T, B, V = 6, 8, 96
    y = torch.randn(T, B, V, generator=g).to(DEV); z = (torch.randn(T, B, V, generator=g) * 2).to(DEV)
    tgt = torch.randint(1, V, (T, B), generator=g); tgt[3:, :3] = 0; tgt = tgt.to(DEV)
    st = torch.cuda.current_stream().cuda_stream

    def run(ys, zs, ts, nval, mult):
        N = ys.shape[0] * ys.shape[1]
        ys, zs, ts = ys.contiguous(), zs.contiguous(), ts.contiguous()
        dy = torch.empty_like(ys); rows = torch.empty(2, N, device=DEV)
        assert lib.b2c_kd_token_loss(ys.data_ptr(), zs.data_ptr(), ts.data_ptr(), N, V, 4.0, 0.5, 0.5, mult, nval.data_ptr(),
                                     dy.data_ptr(), rows[0].data_ptr(), rows[1].data_ptr(), 0, st) == 0
        return dy
    nval = torch.tensor([int((tgt != 0).sum())], dtype=torch.int32, device=DEV)
    full = run(y, z, tgt, nval, 1.0)
    halves = torch.cat([run(y[:, :4], z[:, :4], tgt[:, :4], nval, 2.0), run(y[:, 4:], z[:, 4:], tgt[:, 4:], nval, 2.0)], dim=1) / 2
    assert relerr(halves.cpu(), full.cpu()) < 1e-5


def test_full_size_properties_config2():
    """BASELINE config 2 sizes (B512 T20 V5000, bf16): size-independent properties instead of an oracle run."""
    V, E, H, L, B, T = 5000, 256, 512, 2, 512, 20
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(384, E, seed=1)
    model, projector = build_student(params, pparams, V, E, H, L, True, 384, DEV)
    batch = O.synthetic_batch(B, T, V, E, H, seed=1234)
    got = run_kd_step(model, projector, batch, DEV, torch.bfloat16)
    att = got["attention_weights"]
    assert torch.allclose(att.sum(-1), torch.ones(T, B), atol=1e-4) and (att >= 0).all()
    for k, v in got["grads"].items():
        assert torch.isfinite(v).all(), k
    assert torch.isfinite(got["d_encoder_features"]).all() and all(v == v and v >= 0 for v in got["loss"].values())
    # the same step in fp32 parity mode agrees with bf16 within the bf16 tolerance on the loss
    got32 = run_kd_step(model, projector, batch, DEV, torch.float32)
    for k in got["loss"]:
        assert abs(got["loss"][k] - got32["loss"][k]) <= BF16_TOL * max(abs(got32["loss"][k]), 1e-6), k
    # dlogits rows sum to zero (softmax gradients) -> output bias gradient sums to ~0
    assert abs(float(got32["grads"]["decoder.output_projection.3.bias"].sum())) < 1e-4
    # PAD rows contribute only the KD part: CE weight is ~0 at the defaults, so grads must be independent of targets
    batch2 = dict(batch); batch2["targets"] = batch["targets"].clone().clamp_min(1)
    got_b = run_kd_step(model, projector, batch2, DEV, torch.float32)
    assert relerr(got_b["grads"]["decoder.lstm.weight_hh_l0"], got32["grads"]["decoder.lstm.weight_hh_l0"]) < 1e-5


def test_config2_matches_oracle():
    """The BENCHMARKED configuration (BASELINE configs[1]: B=512, T=20, V=5000, E256/H512/L2, refinement, 197x384 teacher features)
    against the oracle on the same inputs: fp32 mode within 1e-4 and bf16 mode within max(2e-2, 1.2 x autocast-reference error).
    This is where the multi-M-tile BN=128/256 GEMM plans, the split-K plans, the 512-CTA attention waves and (bf16) the persistent
    recurrence kernels of the bench run.  The oracle runs in fp64 on the GPU (plain tensor arithmetic, device-agnostic; ~2 s)."""
    V, E, H, L, B, T = 5000, 256, 512, 2, 512, 20
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(384, E, seed=1)
    batch = O.synthetic_batch(B, T, V, E, H, seed=1234)
    ref = O.kd_step(to_device(params, DEV), to_device(pparams, DEV), to_device(batch, DEV), dtype=torch.float64)
    ref = {k: ({kk: (vv.cpu() if torch.is_tensor(vv) else vv) for kk, vv in v.items()} if isinstance(v, dict) else v.cpu()) for k, v in ref.items()}
    model, projector = build_student(params, pparams, V, E, H, L, True, 384, DEV)
    got32 = run_kd_step(model, projector, batch, DEV, torch.float32)
    # fp32: 1e-4 in the max norm for every tensor, except the gradients that reach back through a ReLU whose pre-activations
    # number 12.8 M (refinement FFN) / 25.8 M (projector) here.  A handful of them lie within fp32 round-off of 0; the mask of such
    # an element differs between ANY two evaluation orders (fp64 oracle vs fp32 kernel, or torch's own fp32 CPU vs GPU), and one
    # flipped element is a whole term of a 25 088-term sum: measured 8e-3 of the largest entry in ONE row of d ffn.0.weight with
    # every other row exact to 1e-6, and a dense 3-5e-4 ripple in what lies upstream of it (LayerNorm 1, the attention block).
    # Those tensors are held to 2e-3 (per-tensor L2) / 2e-2 (max norm); a kernel bug there is an O(1) error.
    relu_upstream = ("grad:attention_refinement.attention.", "grad:attention_refinement.ffn.0.", "grad:attention_refinement.norm1.",
                     "pgrad:feature_projection.0.", "d_encoder_features")
    e_max, e_l2 = step_errors(got32, ref, "max"), step_errors(got32, ref, "l2")
    bad = [(k, e_max[k], e_l2[k]) for k in e_max
           if not ((e_l2[k] < 2e-3 and e_max[k] < 2e-2) if k.startswith(relu_upstream) else e_max[k] < FP32_TOL)]
    assert not bad, bad
    got16 = run_kd_step(model, projector, batch, DEV, torch.bfloat16)
    meta = dict(V=V, E=E, H=H, L=L)
    compare_step_calibrated(got16, ref, autocast_reference_errors(params, pparams, meta, batch, ref, DEV), BF16_TOL)


@pytest.mark.parametrize("fake_dp", [False, True])
def test_graphed_step_equals_eager_step(fake_dp, monkeypatch):
    """GraphedKDStep (one CUDA graph per KD step) reproduces the eagerly issued step: same loss parts, same updated weights.
    fake_dp: the multi-rank control flow on one GPU (two graphs; the count exchange under the forward and the decoder-gradient
    exchange under the refinement backward, tied to the graph by external events) with identities in place of the collectives."""
    if fake_dp:
        monkeypatch.setenv("B2C_FAKE_DP", "1")
    from imagecaptioner_b200.ddp import FlatGradAllReducer
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    V, E, H, L, B, T = 200, 64, 128, 2, 8, 6
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(48, E, seed=1)
    batch = {k: (v.to(DEV) if v is not None else None) for k, v in O.synthetic_batch(B, T, V, E, H, Et=48, seed=7).items()}
    results = []
    for use_graph in (False, True):
        model, projector = build_student(params, pparams, V, E, H, L, True, 48, DEV)
        model.decoder.compute_dtype = torch.float32
        trainable = [p for p in list(model.parameters()) + list(projector.parameters()) if p.requires_grad]
        reducer = FlatGradAllReducer(trainable)
        opt = torch.optim.AdamW(trainable, lr=1e-3, weight_decay=0.01, fused=True, capturable=True)
        kd = GraphedKDStep(model, projector, DistillationLoss(vocab_size=V), opt, reducer, batch, autocast_dtype=None,
                           use_graph=use_graph, warmup_steps=0 if not use_graph else 1)
        if use_graph:      # the warm-up + capture bodies already took 2 optimizer steps on this copy: restart from the same point
            model.load_state_dict({k: v.float() for k, v in params.items()}, strict=False)
            projector.load_state_dict({k: v.float() for k, v in pparams.items()})
            opt.state.clear()
        outs = [kd.step().clone() for _ in range(3)]
        torch.cuda.synchronize()
        results.append((torch.stack(outs).cpu(), {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}))
    (l0, w0), (l1, w1) = results
    assert relerr(l1[0], l0[0]) < 1e-5                       # first step: identical weights, identical loss parts
    assert float(l0[2, 0]) < float(l0[0, 0])                 # and the loss goes down over the three steps
    if fake_dp:
        assert kd.overlap_comm and kd._early is not None     # the overlapped path really ran, on the decoder's gradient segment


@pytest.mark.parametrize("B", [128, 256])
def test_larger_batch_matches_oracle(B):
    """Several M tiles per GEMM and several waves of attention CTAs (and, with B2C_SUB_BATCHES set, the forked sub-batch
    streams): same results as the oracle on the whole batch."""
    V, E, H, L, T = 120, 32, 64, 2, 4
    params = O.init_student_params(V, E, H, L, True, seed=5)
    pparams = O.init_projector_params(24, E, seed=6)
    batch = O.synthetic_batch(B, T, V, E, H, Et=24, seed=8)
    model, projector = build_student(params, pparams, V, E, H, L, True, 24, DEV)
    got = run_kd_step(model, projector, batch, DEV, torch.float32)
    ref = O.kd_step(params, pparams, batch)
    compare_step(got, ref, FP32_TOL, verbose=False)


def test_large_variant_real_dims_fp32_and_bf16():
    """BASELINE config 5 dimensions (E384 H768 3-layer LSTM, V10000, refinement with head_dim 96, identity channel projection
    384 -> 384) at a small batch against the oracle: exercises the E > 256 kernel variants (two LayerNorm chunks per lane,
    three float4 per lane in the attention score phase, 3 stacked fused gate GEMMs)."""
    V, E, H, L, B, T = 10000, 384, 768, 3, 4, 3
    params = O.init_student_params(V, E, H, L, True, seed=11)
    pparams = O.init_projector_params(384, E, seed=12)            # {} : identity projection, pooling only
    batch = O.synthetic_batch(B, T, V, E, H, Et=384, seed=13)
    ref = O.kd_step(params, pparams, batch, dtype=torch.float64)    # fp64 oracle: isolates the kernel error from fp32-CPU noise
    model, projector = build_student(params, pparams, V, E, H, L, True, 384, DEV)
    got = run_kd_step(model, projector, batch, DEV, torch.float32)
    compare_step(got, ref, FP32_TOL, verbose=False)
    got16 = run_kd_step(model, projector, batch, DEV, torch.bfloat16)
    meta = dict(V=V, E=E, H=H, L=L)
    compare_step_calibrated(got16, ref, autocast_reference_errors(params, pparams, meta, batch, ref, DEV), BF16_TOL, verbose=False)
    toks, lens = model.decoder.greedy(model.attention_refinement(batch["encoder_features"].to(DEV)).float(), 6)
    assert tuple(toks.shape) == (6, B) and int(lens.max()) <= 6


def test_validation_path_matches_reference_fixture():
    """validate_student_model on the native path (eval loss without gradients, argmax in the loss pass, device BLEU-1) against the
    reference's loss, `logits.argmax(-1)` and compute_bleu_score on the golden KD case (tests/golden/validation_case.pt)."""
    from imagecaptioner_b200.distillation_utils import DistillationLoss, TeacherWrapper
    from imagecaptioner_b200.validation import validate_student_model
    g = torch.load(os.path.join(GOLDEN, "kd_small_default.pt"), weights_only=False)
    fx = torch.load(os.path.join(GOLDEN, "validation_case.pt"), weights_only=False)["kd_small_default"]
    m, batch = g["meta"], g["batch"]
    Et = batch["teacher_features"].shape[-1]
    model, projector = build_student(g["params"], g["proj_params"], m["V"], m["E"], m["H"], m["L"], m["refinement"], Et, DEV)
    model.decoder.compute_dtype = torch.float32
    model.attention_refinement.compute_dtype = torch.float32
    projector.compute_dtype = torch.float32
    loss_mod = DistillationLoss(m["alpha"], m["beta"], m["gamma"], m["temperature"], vocab_size=m["V"])
    with torch.no_grad():
        logits, enc, hids, _ = model(batch["encoder_features"].to(DEV), batch["captions_input"].to(DEV))
        th = batch["teacher_hiddens"]
        t_out = {"logits": batch["teacher_logits"].to(DEV), "encoder_features": projector(batch["teacher_features"].to(DEV)),
                 "hidden_states": [th[t].to(DEV) for t in range(th.shape[0])]}
        loss, loss_dict, pred = loss_mod.evaluate({"logits": logits, "encoder_features": enc, "hidden_states": hids}, t_out,
                                                  batch["targets"].to(DEV))
    for k, v in g["reference"]["loss"].items():
        assert abs(loss_dict[k] - v) <= 1e-4 * max(1.0, abs(v)), k
    assert torch.equal(pred.cpu().long(), fx["predicted_tokens"])
    from imagecaptioner_b200 import _ops
    assert torch.allclose(_ops.bleu1(pred, batch["targets"].to(DEV)).cpu(), fx["bleu"], atol=1e-6)

    # the whole function, with a stub teacher that replays the fixture's teacher outputs (hidden_states None like TeacherWrapper)
    class StubTeacher(TeacherWrapper):
        def __init__(self):
            torch.nn.Module.__init__(self)
        def forward(self, images, captions):
            return {"logits": batch["teacher_logits"].to(DEV), "encoder_features": batch["teacher_features"].to(DEV), "hidden_states": None}
    captions = torch.cat([batch["captions_input"][:1], batch["targets"]], dim=0)          # (T+1, B): input = [:-1], target = [1:]
    captions[:-1] = batch["captions_input"]
    loader = [(batch["encoder_features"], captions)] * 3
    avg_loss, avg_bleu = validate_student_model(model, StubTeacher(), loader, loss_mod, {"encoder": projector}, DEV, vocab=None, max_batches=2)
    ref = O.kd_step(g["params"], g["proj_params"], dict(batch, teacher_hiddens=None), m["alpha"], m["beta"], m["gamma"], m["temperature"])
    assert abs(avg_loss - ref["loss"]["total_loss"]) <= 1e-4 * max(1.0, abs(ref["loss"]["total_loss"]))
    assert abs(avg_bleu - float(fx["bleu"][:2].mean())) < 1e-6
    assert not model.training


def test_fused_argmax_decode_equals_logits_path(tmp_path):
    """bf16 greedy decode with the argmax reduced inside the vocabulary-head GEMM epilogue (no logits written) gives exactly the
    tokens and lengths of the logits + argmax-kernel path (B2C_DECODE_LOGITS=1), including an edge N tile (V = 5000) and a batch
    that is not a multiple of the 128-row tile."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = []
    for mode in ("fused", "logits"):
        env = dict(os.environ)
        env.pop("B2C_DECODE_LOGITS", None)
        if mode == "logits":
            env["B2C_DECODE_LOGITS"] = "1"
        out = str(tmp_path / f"tok_{mode}.pt")
        r = subprocess.run([sys.executable, os.path.join(root, "tools", "check_decode_argmax.py"), out], env=env, cwd=root,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(torch.load(out))
    assert torch.equal(outs[0]["tokens"], outs[1]["tokens"])
    assert torch.equal(outs[0]["lengths"], outs[1]["lengths"])
    assert outs[0]["tokens"].unique().numel() > 8              # not a degenerate caption (19 distinct ids over columns 171..4393)


@pytest.mark.parametrize("V,B,T", [(5000, 96, 7), (1000, 33, 3)])
def test_logits_free_validation_matches_logits_path_and_oracle(V, B, T):
    """b2c_decoder_forward_eval (SURVEY.md section 8f row 4): the vocabulary-head GEMM's epilogue reduces its tiles to per-row partials
    of the token-KD / CE terms and the argmax against the teacher logits, so validation never materialises the (T,B,V) logits.
    Against (i) the fp64 oracle (loss parts, predictions where the oracle's top-2 margin is not a rounding tie) and (ii) the bf16
    logits path `DistillationLoss.evaluate` on the same inputs.  V = 5000: an edge N tile; B*T not a multiple of the 128-row tile."""
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    E, H, L = 64, 128, 2
    params = O.init_student_params(V, E, H, L, True, seed=21, logit_scale=6.0)
    pparams = O.init_projector_params(48, E, seed=22)
    batch = O.synthetic_batch(B, T, V, E, H, Et=48, seed=23)
    ref = O.kd_step(to_device(params, DEV), to_device(pparams, DEV), to_device(batch, DEV), dtype=torch.float64)
    model, projector = build_student(params, pparams, V, E, H, L, True, 48, DEV)
    model.decoder.compute_dtype = torch.bfloat16
    model.attention_refinement.compute_dtype = torch.bfloat16
    projector.compute_dtype = torch.bfloat16
    assert model.supports_fused_validation()
    loss_mod = DistillationLoss(0.5, 0.2, 0.1, 4.0, vocab_size=V)          # CE weight 0.2: the CE partials matter
    dev_b = to_device(batch, DEV)
    th = dev_b["teacher_hiddens"]
    with torch.no_grad():
        t_out = {"logits": dev_b["teacher_logits"], "encoder_features": projector(dev_b["teacher_features"]),
                 "hidden_states": [th[t] for t in range(th.shape[0])]}
        _, fused, pred_f = loss_mod.evaluate_fused(model, dev_b["encoder_features"], dev_b["captions_input"], t_out, dev_b["targets"])
        logits, enc, hids, _ = model(dev_b["encoder_features"], dev_b["captions_input"])
        _, unfused, pred_u = loss_mod.evaluate({"logits": logits, "encoder_features": enc, "hidden_states": hids}, t_out, dev_b["targets"])
    ref_loss = O.kd_step(params, pparams, batch, 0.5, 0.2, 0.1, 4.0)["loss"]
    for k, v in ref_loss.items():
        assert abs(fused[k] - v) <= BF16_TOL * max(abs(v), 1e-6), (k, fused[k], v)
        assert abs(fused[k] - unfused[k]) <= 5e-3 * max(abs(v), 1e-6), (k, fused[k], unfused[k])
    # predictions: identical to the oracle's argmax wherever its top-2 margin exceeds bf16-mode noise; the fused path keeps the
    # fp32 accumulators, the logits path rounds them to bf16 first, so the two may differ on near-ties only
    y = ref["logits"].double()
    top2 = y.topk(2, dim=-1).values
    clear = ((top2[..., 0] - top2[..., 1]) > 2e-2 * y.abs().amax()).cpu()
    oracle_pred = y.argmax(-1).cpu()
    assert int(clear.sum()) >= 10
    assert torch.equal(pred_f.cpu().long()[clear], oracle_pred[clear])
    assert float((pred_f.cpu().long() == oracle_pred).float().mean()) > 0.9
    assert float((pred_f == pred_u).float().mean()) > 0.97


def test_cluster_recurrence_kernel_matches_per_step_kernels():
    """The opt-in cluster forward recurrence (csrc/recur_cluster.cuh, B2C_CLUSTER=1) against the per-step kernels on the same bf16 KD
    step: every output and gradient within 2e-2 (L2) at batch sizes that give 1 cluster with idle CTAs (16), ragged 35-row slices with
    an empty CTA (70 -> 3 clusters) and several clusters (240).  The switch is read once per process, hence the subprocesses."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "cluster_ab.py"), "16", "70", "240"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "cluster A/B: OK" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]


def test_decoder_forward_with_initial_hidden_state_matches_reference():
    """LSTMDecoder.forward(image_features, captions, hidden=(h0, c0)) (reference src/student_model.py:205, :219-222): outputs, hidden
    states, attention weights and every gradient against the REFERENCE's own run (tests/golden/hidden_init_case.pt, generator
    oracle/pin_hidden.py), fp32 <= 1e-4; bf16 within 2e-2 (L2); with and without the split (prepared) forward."""
    g = torch.load(os.path.join(GOLDEN, "hidden_init_case.pt"), weights_only=False)
    m, ref = g["meta"], g["reference"]
    model, _ = build_student(g["params"], {}, m["V"], m["E"], m["H"], m["L"], False, m["E"], DEV)
    dec = model.decoder
    cap = g["captions"].to(DEV)
    hidden = (g["h0"].to(DEV), g["c0"].to(DEV))
    for dtype, tol, metric in ((torch.float32, FP32_TOL, relerr), (torch.bfloat16, 2e-2, relerr_l2)):
        for split in (False, True):
            dec.compute_dtype = dtype
            dec.zero_grad(set_to_none=True)
            f = g["feats"].to(DEV).clone().requires_grad_(True)
            prepared = dec.prepare(cap, m["S"]) if split else None
            out, hids, atts = dec(f, cap, hidden, prepared=prepared)
            (out.float() * g["dout"].to(DEV)).sum().backward()
            assert metric(out.float().cpu(), ref["outputs"]) < tol
            assert metric(torch.stack(list(hids)).float().cpu(), ref["hidden_states"]) < tol
            assert metric(torch.stack(atts).float().cpu(), ref["attention_weights"]) < tol
            assert metric(f.grad.float().cpu(), ref["d_feats"]) < tol
            for k, v in ref["grads"].items():
                got = dict(model.named_parameters())[k].grad.float().cpu()
                assert metric(got, v) < (tol if dtype == torch.float32 else 4e-2), (k, str(dtype), metric(got, v))
    with pytest.raises(NotImplementedError):
        dec(g["feats"].to(DEV), cap, (hidden[0].clone().requires_grad_(True), hidden[1]))
    with pytest.raises(ValueError):
        dec(g["feats"].to(DEV), cap, (hidden[0][:1], hidden[1][:1]))


@pytest.mark.parametrize("env,tol", [("B2C_MERGE_REC=1,0", 2e-2), ("B2C_BG_CTAS=10,0", 1.5e-2), ("B2C_POST_OCC3=1,0", 1.5e-2)])
def test_ab_switches_keep_the_results(env, tol):
    """Every performance switch that changes the dataflow of the default bf16 path leaves the KD step's outputs and gradients where
    they were (per-tensor relative L2; not bit-identical: the contraction order changes, and the K-split reductions are fp32 atomics whose
    order varies from run to run -- two runs of the SAME build differ by up to ~8e-3 on the smallest gradients in bf16 mode): the top
    layer's recurrent half merged into
    the query-projection GEMM, the background CTA budget (changes the split-K plans of the capped GEMMs), the attn_post register variant."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "cluster_ab.py"), "--env", env, "--tol", str(tol), "48", "512"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "A/B: OK" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
