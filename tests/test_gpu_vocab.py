"""GPU: bf16 throughput mode for vocabulary sizes that are not a multiple of 8 (what the reference's frequency-thresholded
Vocabulary produces).  The logits gradient lives at row pitch roundup(V, 8): the token pass streams unaligned rows through its
TMA pipeline and the vocabulary head's backward contractions stay on tensor cores."""
import pytest
import torch

from oracle import kd_oracle as O
from oracle import manual_backward as M
from tests.harness import (autocast_reference_errors, build_student, compare_step, compare_step_calibrated, relerr, relerr_l2, run_kd_step,
                           to_device)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _lib():
    from imagecaptioner_b200 import _ops
    return _ops, _ops.load_library()


def _pitched_token_loss(yd, zd, td, V, temp, alpha, w_ce):
    """b2c_kd_token_loss_pitched on (N, V) logits -> (row_kl, row_ce, n_valid, padded dlogits buffer (N, Vp))."""
    ops, lib = _lib()
    N = td.numel()
    Vp = (V + 7) // 8 * 8
    st = torch.cuda.current_stream().cuda_stream
    nval = torch.zeros(1, dtype=torch.int32, device=DEV)
    assert lib.b2c_count_valid(td.data_ptr(), N, V, nval.data_ptr(), st) == 0
    dy = torch.full((N, Vp), float("nan"), dtype=torch.bfloat16, device=DEV)      # every written column is checked below
    rows = torch.empty(2, N, device=DEV)
    rc = lib.b2c_kd_token_loss_pitched(yd.data_ptr(), zd.data_ptr(), td.data_ptr(), N, V, temp, alpha, w_ce, 1.0, nval.data_ptr(),
                                       dy.data_ptr(), Vp, rows[0].data_ptr(), rows[1].data_ptr(), ops.B2C_BF16, st)
    assert rc == 0, lib.b2c_last_error()
    torch.cuda.synchronize()
    return rows[0].cpu(), rows[1].cpu(), int(nval.item()), dy


@pytest.mark.parametrize("V", [4999, 5001, 1001, 203, 57])
@pytest.mark.parametrize("temp", [4.0, 2.0])
def test_unaligned_token_pass(V, temp):
    g = torch.Generator().manual_seed(V)
    T, B = 7, 9
    N = T * B
    y = (torch.randn(T, B, V, generator=g) * 1.5).bfloat16()
    z = torch.randn(T, B, V, generator=g) * 2.0
    tgt = torch.randint(1, V, (T, B), generator=g)
    tgt[-2:, ::2] = 0                                        # PAD rows
    alpha, w_ce = 0.6, 0.25
    yd, zd, td = y.to(DEV), z.to(DEV), tgt.to(DEV)
    kl, ce, nval, dy = _pitched_token_loss(yd, zd, td, V, temp, alpha, w_ce)
    assert nval == int((tgt != 0).sum())
    yy, zz = y.double(), z.double()
    kd = temp * temp * kl.double().sum() / N
    assert abs(kd - O.token_kd(yy, zz, temp)) < 1e-4 * abs(float(O.token_kd(yy, zz, temp))) + 1e-7
    ce_ref = O.cross_entropy_ignore_pad(yy, tgt)
    assert abs(ce.double().sum() / nval - ce_ref) < 1e-4 * abs(float(ce_ref))
    gref = M.kd_token_grad(yy, zz, tgt, temp, alpha, w_ce)
    assert relerr(dy[:, :V].float().cpu().view(T, B, V), gref) < 8e-3
    assert torch.equal(dy[:, V:].cpu(), torch.zeros(N, dy.shape[1] - V, dtype=torch.bfloat16))     # exact zeros, no NaN left

    # logits that are views ending exactly at the end of their storage (the last rows' 16-byte ranges would run past it), one of
    # them starting 3 elements into a 16-byte word (the first row's range would start before it): the rows that are read with
    # plain loads give the same results as the bulk-copied rows of a fresh tensor
    for off in (8, 3):
        ys = torch.empty(N * V + off, dtype=torch.bfloat16, device=DEV)
        yv = ys.narrow(0, off, N * V).view(N, V)
        yv.copy_(yd.view(N, V))
        zs = torch.empty(N * V + 1, device=DEV)
        zv = zs.narrow(0, 1, N * V).view(N, V)
        zv.copy_(zd.view(N, V))
        kl2, ce2, _, dy2 = _pitched_token_loss(yv, zv, td, V, temp, alpha, w_ce)
        assert torch.equal(kl2, kl) and torch.equal(ce2, ce) and torch.equal(dy2, dy)


def test_unaligned_token_pass_all_pad():
    g = torch.Generator().manual_seed(3)
    V = 203
    y = torch.randn(3, 4, V, generator=g).bfloat16().to(DEV)
    kl, ce, nval, dy = _pitched_token_loss(y, y.float(), torch.zeros(3, 4, dtype=torch.long, device=DEV), V, 4.0, 1.0, 0.0)
    assert nval == 0 and float(kl.abs().max()) < 1e-5 and float(ce.abs().max()) == 0.0      # KL(p||p) = 0, CE 0 on PAD rows
    assert torch.isfinite(dy.float()).all() and float(dy.float().abs().max()) < 1e-5


def test_pitched_entries_reject_bad_pitch():
    ops, lib = _lib()
    y = torch.zeros(4, 203, dtype=torch.bfloat16, device=DEV)
    z = torch.zeros(4, 203, device=DEV)
    t = torch.ones(4, dtype=torch.long, device=DEV)
    n = torch.ones(1, dtype=torch.int32, device=DEV)
    rows = torch.empty(2, 4, device=DEV)
    dy = torch.empty(4, 212, dtype=torch.bfloat16, device=DEV)
    for ld, dt in ((100, ops.B2C_BF16), (210, ops.B2C_BF16), (208, ops.B2C_F32)):       # < V, not a multiple of 8, fp32
        rc = lib.b2c_kd_token_loss_pitched(y.data_ptr(), z.data_ptr(), t.data_ptr(), 4, 203, 4.0, 0.5, 0.5, 1.0, n.data_ptr(), dy.data_ptr(),
                                           ld, rows[0].data_ptr(), rows[1].data_ptr(), dt, torch.cuda.current_stream().cuda_stream)
        err = lib.b2c_last_error()
        assert rc == -1 and (b"ld_dlogits" in err or b"pitch" in err), (ld, dt, err)          # B2C_EINVAL


def _problem(V, B, T, E=32, H=64, L=2, Et=24, seed=5):
    params = O.init_student_params(V, E, H, L, True, seed=seed)
    pparams = O.init_projector_params(Et, E, seed=seed + 1)
    batch = O.synthetic_batch(B, T, V, E, H, Et=Et, seed=seed + 3)
    return params, pparams, batch, dict(V=V, E=E, H=H, L=L), Et


def test_kd_step_v4999_bf16_and_fp32_match_oracle():
    """The whole KD step at V = 4999 with B = 256 (multi-tile head GEMMs): bf16 within max(2e-2, 1.2 x the autocast reference's
    error) of the fp64 oracle, fp32 within 1e-4."""
    params, pparams, batch, meta, Et = _problem(4999, 256, 4)
    ref = O.kd_step(to_device(params, DEV), to_device(pparams, DEV), to_device(batch, DEV), dtype=torch.float64)
    ref = {k: ({kk: (vv.cpu() if torch.is_tensor(vv) else vv) for kk, vv in v.items()} if isinstance(v, dict) else v.cpu()) for k, v in ref.items()}
    model, projector = build_student(params, pparams, meta["V"], meta["E"], meta["H"], meta["L"], True, Et, DEV)
    got16 = run_kd_step(model, projector, batch, DEV, torch.bfloat16)
    compare_step_calibrated(got16, ref, autocast_reference_errors(params, pparams, meta, batch, ref, DEV), 2e-2, verbose=False)
    got32 = run_kd_step(model, projector, batch, DEV, torch.float32)
    compare_step(got32, ref, 1e-4, verbose=False)


def _kernel_names(V, B=256, T=4):
    params, pparams, batch, meta, Et = _problem(V, B, T)
    model, projector = build_student(params, pparams, V, meta["E"], meta["H"], meta["L"], True, Et, DEV)
    run_kd_step(model, projector, batch, DEV, torch.bfloat16)                  # warm-up: module loads outside the trace
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_kd_step(model, projector, batch, DEV, torch.bfloat16)
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_v4999_step_runs_no_fallback_kernels():
    names = _kernel_names(4999)
    assert not [n for n in names if "gemm_simt_kernel" in n or "kd_token_loss_kernel" in n], sorted(set(names))
    assert any("kd_token_loss_pipe_unaligned_kernel" in n for n in names)
    assert any("colsum_vec_pitched_kernel" in n for n in names)
    aligned = _kernel_names(5000)                                              # V % 8 == 0: none of the new kernels
    assert not [n for n in aligned if "unaligned" in n or "pitched" in n]
    assert any("kd_token_loss_pipe_kernel" in n for n in aligned)


def test_layout_fallback_extra_term_on_outputs():
    """The decoder's backward takes the padded logits gradient with its pitch, and any other layout contiguous.  Both give the
    gradients of the same logits gradient forced into the contiguous layout (a hook on `outputs`): for the KD loss alone (the
    padded view reaches the decoder) and with an extra term on `outputs` (autograd sums two gradients of the logits first)."""
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    V, B, T = 4999, 64, 4
    params, pparams, batch, meta, Et = _problem(V, B, T)
    model, projector = build_student(params, pparams, V, meta["E"], meta["H"], meta["L"], True, Et, DEV)
    for m in (model.decoder, model.attention_refinement, projector):
        m.compute_dtype = torch.bfloat16
    d = to_device(batch, DEV)
    loss_mod = DistillationLoss(0.7, 0.2, 0.1, 4.0, vocab_size=V)
    t_out = {"logits": d["teacher_logits"], "encoder_features": projector(d["teacher_features"]).detach(),
             "hidden_states": [d["teacher_hiddens"][t] for t in range(d["teacher_hiddens"].shape[0])]}
    w = torch.randn(T, B, V, generator=torch.Generator().manual_seed(9)).to(DEV)
    seen = []

    def grads(extra, force_contiguous):
        model.zero_grad(set_to_none=True)
        outputs, enc, hids, _ = model(d["encoder_features"], d["captions_input"])
        outputs.register_hook(lambda g: seen.append((g.stride(), float(g.float().pow(2).mean().sqrt()))) or
                              (g.contiguous() if force_contiguous else None))
        loss = loss_mod({"logits": outputs, "encoder_features": enc, "hidden_states": hids}, t_out, d["targets"])[0]
        if extra:
            loss = loss + (outputs.float() * w).sum()
        loss.backward()
        torch.cuda.synchronize()
        return {k: p.grad.detach().double().cpu() for k, p in model.named_parameters() if p.grad is not None}

    g_kd = grads(False, False)
    assert seen[-1][0][1] == (V + 7) // 8 * 8                   # the KD term alone hands the decoder the padded view
    w *= seen[-1][1]                                            # the extra term's logits gradient: the KD term's RMS
    g_kd_ref = grads(False, True)
    g_both = grads(True, False)
    g_both_ref = grads(True, True)
    for k in g_kd:
        assert relerr_l2(g_kd[k], g_kd_ref[k]) < 1e-2, k
        assert relerr_l2(g_both[k], g_both_ref[k]) < 1e-2, k
    k = "decoder.output_projection.3.weight"
    assert relerr_l2(g_both[k], g_kd[k]) > 2e-2                 # the extra term is in the gradient


def test_fused_validation_v4999_matches_logits_path():
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    V, B, T = 4999, 33, 3
    E, H, L, Et = 64, 128, 2, 48
    params = O.init_student_params(V, E, H, L, True, seed=21, logit_scale=6.0)
    pparams = O.init_projector_params(Et, E, seed=22)
    batch = O.synthetic_batch(B, T, V, E, H, Et=Et, seed=23)
    model, projector = build_student(params, pparams, V, E, H, L, True, Et, DEV)
    for m in (model.decoder, model.attention_refinement, projector):
        m.compute_dtype = torch.bfloat16
    assert model.supports_fused_validation()
    loss_mod = DistillationLoss(0.5, 0.2, 0.1, 4.0, vocab_size=V)
    d = to_device(batch, DEV)
    with torch.no_grad():
        t_out = {"logits": d["teacher_logits"], "encoder_features": projector(d["teacher_features"]),
                 "hidden_states": [d["teacher_hiddens"][t] for t in range(d["teacher_hiddens"].shape[0])]}
        _, fused, pred_f = loss_mod.evaluate_fused(model, d["encoder_features"], d["captions_input"], t_out, d["targets"])
        logits, enc, hids, _ = model(d["encoder_features"], d["captions_input"])
        _, unfused, pred_u = loss_mod.evaluate({"logits": logits, "encoder_features": enc, "hidden_states": hids}, t_out, d["targets"])
    for k, v in unfused.items():
        assert abs(fused[k] - v) <= 1e-3 * max(abs(v), 1e-6), (k, fused[k], v)
    # argmax: identical wherever the bf16 logits' top-1 / top-2 margin is at least two bf16 ulps of the top-1 value (rounding the
    # fp32 accumulators to bf16 moves each by at most half an ulp, so the order of those two cannot change)
    top2 = logits.float().topk(2, dim=-1).values
    ulp = torch.exp2(torch.floor(torch.log2(top2[..., 0].abs().clamp_min(1e-30))) - 7)
    clear = (top2[..., 0] - top2[..., 1]) >= 2 * ulp
    assert int(clear.sum()) >= 0.5 * clear.numel()
    assert torch.equal(pred_f[clear].long(), pred_u[clear].long())


def test_graphed_step_v4999_equals_eager_step():
    """GraphedKDStep in bf16 mode at V = 4999 (padded logits gradient inside the captured graph) reproduces the eager step."""
    from imagecaptioner_b200.ddp import FlatGradAllReducer
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    V, E, H, L, B, T = 4999, 64, 128, 2, 8, 6
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(48, E, seed=1)
    batch = {k: (v.to(DEV) if v is not None else None) for k, v in O.synthetic_batch(B, T, V, E, H, Et=48, seed=7).items()}
    results = []
    for use_graph in (False, True):
        model, projector = build_student(params, pparams, V, E, H, L, True, 48, DEV)
        for m in (model.decoder, model.attention_refinement, projector):
            m.compute_dtype = torch.bfloat16
        trainable = [p for p in list(model.parameters()) + list(projector.parameters()) if p.requires_grad]
        reducer = FlatGradAllReducer(trainable)
        opt = torch.optim.AdamW(trainable, lr=1e-3, weight_decay=0.01, fused=True, capturable=True)
        kd = GraphedKDStep(model, projector, DistillationLoss(vocab_size=V), opt, reducer, batch, autocast_dtype=None,
                           use_graph=use_graph, warmup_steps=0 if not use_graph else 1)
        if use_graph:
            model.load_state_dict({k: v.float() for k, v in params.items()}, strict=False)
            projector.load_state_dict({k: v.float() for k, v in pparams.items()})
            opt.state.clear()
        outs = [kd.step().clone() for _ in range(3)]
        torch.cuda.synchronize()
        results.append(torch.stack(outs).cpu())
    l0, l1 = results
    assert relerr(l1[0], l0[0]) < 1e-5                       # first step: identical weights, identical loss parts
    assert relerr(l1, l0) < 2e-2                             # later steps: the same updates up to bf16 reduction order
    assert float(l0[2, 0]) < float(l0[0, 0])
