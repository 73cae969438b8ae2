"""GPU: variable-length batches through one capture.  The *_steps entry points take a device step count n <= T: the decoder
recurrences skip the steps past it, the loss ignores their rows, and the result is that of the n-step batch.  Each test poisons
what must not be read (NaN logits / hidden states past the step count, a 0xFF workspace) and compares with the plain call on
the n-step prefix."""
import ctypes

import pytest
import torch

from oracle import kd_oracle as O
from tests.harness import build_student, relerr, relerr_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _lib():
    from imagecaptioner_b200 import _ops
    return _ops, _ops.load_library()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _steps(n):
    return torch.full((1,), n, dtype=torch.int32, device=DEV)


# ------------------------------------------------------------------ 1. token pass
@pytest.mark.parametrize("V", [5000, 4999, 203, 57])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_token_pass_steps(V, mode):
    ops, lib = _lib()
    Tc, B = 6, 8
    N = Tc * B
    cdt, code = (torch.bfloat16, ops.B2C_BF16) if mode == "bf16" else (torch.float32, ops.B2C_F32)
    ld = (V + 7) // 8 * 8 if (mode == "bf16" and V % 8) else V          # the pitch KDLossFunction uses
    g = torch.Generator().manual_seed(V)
    y = (torch.randn(Tc, B, V, generator=g) * 1.5).to(cdt).to(DEV)
    z = (torch.randn(Tc, B, V, generator=g) * 2.0).to(DEV)
    tgt = torch.randint(1, V, (Tc, B), generator=g).to(DEV)
    tgt[:, ::3] = 0                                                   # PAD rows inside the batch too
    alpha, w_ce, temp = 0.6, 0.25, 4.0
    for Ta in (1, 3, 6):
        n = Ta * B
        t = tgt.clone()
        t[Ta:] = 0                                                    # the caller's contract: PAD past the step count
        yp, zp = y.clone(), z.clone()
        yp[Ta:] = float("nan")                                        # never used
        zp[Ta:] = float("nan")
        nval = ops.count_valid(t, V)
        # reference: the existing entry point on the Ta-step slice
        dy_ref = torch.full((n, ld), float("nan"), dtype=cdt, device=DEV)
        rows_ref = torch.empty(2, n, device=DEV)
        if ld != V:
            rc = lib.b2c_kd_token_loss_pitched(y.data_ptr(), z.data_ptr(), t.data_ptr(), n, V, temp, alpha, w_ce, 1.0, nval.data_ptr(),
                                               dy_ref.data_ptr(), ld, rows_ref[0].data_ptr(), rows_ref[1].data_ptr(), code, _st())
        else:
            rc = lib.b2c_kd_token_loss(y.data_ptr(), z.data_ptr(), t.data_ptr(), n, V, temp, alpha, w_ce, 1.0, nval.data_ptr(),
                                       dy_ref.data_ptr(), rows_ref[0].data_ptr(), rows_ref[1].data_ptr(), code, _st())
        assert rc == 0, lib.b2c_last_error()
        dy = torch.full((N, ld), float("nan"), dtype=cdt, device=DEV)
        rows = torch.full((2, N), float("nan"), device=DEV)
        rc = lib.b2c_kd_token_loss_steps(yp.data_ptr(), zp.data_ptr(), t.data_ptr(), N, V, temp, alpha, w_ce, 1.0, nval.data_ptr(),
                                         dy.data_ptr(), ld, rows[0].data_ptr(), rows[1].data_ptr(), code, _steps(Ta).data_ptr(), B, _st())
        assert rc == 0, lib.b2c_last_error()
        torch.cuda.synchronize()
        w = ld if ld != V else V
        a, b = dy[:n, :w].float(), dy_ref[:, :w].float()
        ulp = 2.0 ** -7 if mode == "bf16" else 2.0 ** -22                 # a few ulp for the scale formed on the device
        assert bool(((a - b).abs() <= 4 * ulp * b.abs() + 1e-30).all()), (Ta, float((a - b).abs().max()))
        assert torch.allclose(rows[:, :n], rows_ref, rtol=1e-6, atol=1e-7), Ta
        assert torch.equal(dy[n:].float().cpu(), torch.zeros(N - n, ld)), Ta           # exact zeros, padding columns included
        assert torch.equal(rows[:, n:].cpu(), torch.zeros(2, N - n)), Ta


# ------------------------------------------------------------------ 2. aux + finalize
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_aux_and_finalize_steps(mode):
    ops, lib = _lib()
    Tc, B, H, E, Ss, St = 6, 8, 64, 32, 10, 12
    N = Tc * B
    cdt, code = (torch.bfloat16, ops.B2C_BF16) if mode == "bf16" else (torch.float32, ops.B2C_F32)
    g = torch.Generator().manual_seed(11)
    fs = torch.randn(B, Ss, E, generator=g).to(DEV)
    ft = torch.randn(B, St, E, generator=g).to(DEV)
    hs = torch.randn(Tc, B, H, generator=g).to(cdt).to(DEV)
    ht = torch.randn(Tc, B, H, generator=g).to(DEV)
    kl = torch.rand(N, generator=g).to(DEV)
    ce = torch.rand(N, generator=g).to(DEV)
    tgt = torch.randint(1, 50, (Tc, B), generator=g).to(DEV)
    beta, gamma, temp, alpha, w_ce = 0.2, 0.1, 4.0, 0.6, 0.1
    fcode = ops.B2C_F32

    def run(T, hs_, ht_, rows_kl, rows_ce, steps):
        dfs = torch.empty(B, Ss, E, device=DEV)
        dft = torch.empty(B, St, E, device=DEV)
        dhs = torch.full((T, B, H), float("nan"), dtype=cdt, device=DEV)
        fp = torch.empty(B, 2, device=DEV)
        hp = torch.full((T * B, 2), float("nan"), device=DEV)
        out5 = torch.empty(5, device=DEV)
        nval = ops.count_valid(tgt[:T] if steps is None else tgt_c, 50)
        aux = (fs.data_ptr(), ft.data_ptr(), B, Ss, St, E, hs_.data_ptr(), ht_.data_ptr(), T, T, H, beta, gamma, dfs.data_ptr(),
               dft.data_ptr(), dhs.data_ptr(), fp.data_ptr(), hp.data_ptr(), code, fcode)
        fin = (rows_kl.data_ptr(), rows_ce.data_ptr(), T * B, nval.data_ptr(), 1.0, fp.data_ptr(), B, E, hp.data_ptr(), T, H, temp, alpha,
               beta, gamma, w_ce, out5.data_ptr())
        if steps is None:
            assert lib.b2c_aux_loss(*aux, _st()) == 0, lib.b2c_last_error()
            assert lib.b2c_loss_finalize(*fin, _st()) == 0, lib.b2c_last_error()
        else:
            assert lib.b2c_aux_loss_steps(*aux, steps.data_ptr(), _st()) == 0, lib.b2c_last_error()
            assert lib.b2c_loss_finalize_steps(*fin, steps.data_ptr(), _st()) == 0, lib.b2c_last_error()
        torch.cuda.synchronize()
        return out5.cpu(), dhs.float().cpu(), dfs.cpu()

    for Ta in (1, 3, 6):
        n = Ta * B
        tgt_c = tgt.clone()
        tgt_c[Ta:] = 0
        hs_p, ht_p = hs.clone(), ht.clone()
        hs_p[Ta:] = float("nan")
        ht_p[Ta:] = float("nan")
        kl_p, ce_p = kl.clone(), ce.clone()
        kl_p[n:] = 0                                                  # what the token pass leaves past the step count
        ce_p[n:] = 0
        ref5, ref_dh, ref_dfs = run(Ta, hs[:Ta].contiguous(), ht[:Ta].contiguous(), kl[:n].contiguous(), ce[:n].contiguous(), None)
        got5, got_dh, got_dfs = run(Tc, hs_p, ht_p, kl_p, ce_p, _steps(Ta))
        assert relerr(got5, ref5) < 1e-6, (Ta, got5, ref5)
        assert torch.equal(got_dh[:Ta], ref_dh), Ta
        assert torch.equal(got_dh[Ta:], torch.zeros(Tc - Ta, B, H)), Ta
        assert torch.equal(got_dfs, ref_dfs)


# ------------------------------------------------------------------ 3. decoder forward + backward
def _decoder_call(shape, code, prm, feats, cap, dlogits, ld, dhid, grads, ws, drop, steps):
    """forward + backward through the C ABI (steps None: the plain entry points) -> (logits, hidden_top, grads, dfeats)."""
    ops, lib = _lib()
    T, B, V, H, S, E = shape.T, shape.B, shape.V, shape.H, shape.S, shape.E
    cdt = torch.bfloat16 if code == ops.B2C_BF16 else torch.float32
    logits = torch.empty(T, B, V, dtype=cdt, device=DEV)
    hid = torch.empty(T, B, H, dtype=cdt, device=DEV)
    attw = torch.empty(T, B, S, device=DEV)
    dfeats = torch.empty(B, S, E, device=DEV)
    fwd = (ctypes.byref(shape), ctypes.byref(prm), feats.data_ptr(), cap.data_ptr(), logits.data_ptr(), hid.data_ptr(), attw.data_ptr(),
           ws.data_ptr(), ws.numel(), code, ctypes.byref(drop))
    grd = ops._fill_struct(ops.B2CGrads(), grads, shape.L)
    if steps is None:
        assert lib.b2c_decoder_forward(*fwd, _st()) == 0, lib.b2c_last_error()
        assert lib.b2c_decoder_backward_pitched(ctypes.byref(shape), ctypes.byref(prm), feats.data_ptr(), cap.data_ptr(), hid.data_ptr(),
                                                attw.data_ptr(), dlogits.data_ptr(), ld, dhid.data_ptr(), ctypes.byref(grd), dfeats.data_ptr(),
                                                ws.data_ptr(), ws.numel(), code, ctypes.byref(drop), 0, _st()) == 0, lib.b2c_last_error()
    else:
        assert lib.b2c_decoder_forward_steps(*fwd, steps.data_ptr(), _st()) == 0, lib.b2c_last_error()
        assert lib.b2c_decoder_backward_steps(ctypes.byref(shape), ctypes.byref(prm), feats.data_ptr(), cap.data_ptr(), hid.data_ptr(),
                                              attw.data_ptr(), dlogits.data_ptr(), ld, dhid.data_ptr(), ctypes.byref(grd), dfeats.data_ptr(),
                                              ws.data_ptr(), ws.numel(), code, ctypes.byref(drop), 0, steps.data_ptr(), _st()) == 0, lib.b2c_last_error()
    torch.cuda.synchronize()
    return logits, hid, [t.detach().double().cpu() for t in grads], dfeats.double().cpu()


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("L,p", [(1, 0.0), (2, 0.3)])
def test_decoder_steps_match_prefix(mode, L, p):
    """Forward + backward at T_cap with a step count == the plain calls at T = T_act on the same features and caption prefix, with
    the workspace pre-filled with 0xFF bytes (NaN) so that the finite saves (I2) and zero gradient rows (I3) are exercised."""
    ops, lib = _lib()
    V, E, H, B, S, Tc = 203, 32, 64, 16, 10, 6
    cdt, code = (torch.bfloat16, ops.B2C_BF16) if mode == "bf16" else (torch.float32, ops.B2C_F32)
    ld = (V + 7) // 8 * 8 if mode == "bf16" else V
    params = O.init_student_params(V, E, H, L, True, seed=3)
    master = [params["decoder." + k].float().contiguous().to(DEV) for k in ops.param_order(L)]
    prm = ops._fill_struct(ops.B2CParams(), master, L)
    g = torch.Generator().manual_seed(4)
    feats = torch.randn(B, S, E, generator=g).to(cdt).to(DEV)
    cap = torch.randint(1, V, (Tc, B), generator=g).to(DEV)
    dl = (torch.randn(Tc, B, V, generator=g) * 1e-2).to(cdt)
    dh = (torch.randn(Tc, B, H, generator=g) * 1e-2).to(cdt)
    drop = ops.B2CDropout(p, 1234, None)
    for Ta in (1, Tc // 2, Tc):
        ref_shape = ops.B2CShape(B, Ta, S, E, H, L, V)
        ws_ref = torch.full((ops.workspace_bytes(ref_shape, code, ops.B2C_WS_TRAIN),), 0xFF, dtype=torch.uint8, device=DEV)
        dl_ref = torch.zeros(Ta, B, ld, dtype=cdt, device=DEV)
        dl_ref[..., :V] = dl[:Ta].to(DEV)
        grads_ref = [torch.empty_like(m) for m in master]
        lo_ref, hid_ref, g_ref, df_ref = _decoder_call(ref_shape, code, prm, feats, cap[:Ta].contiguous(), dl_ref, ld, dh[:Ta].to(DEV).contiguous(),
                                                       grads_ref, ws_ref, drop, None)
        shape = ops.B2CShape(B, Tc, S, E, H, L, V)
        ws = torch.full((ops.workspace_bytes(shape, code, ops.B2C_WS_TRAIN),), 0xFF, dtype=torch.uint8, device=DEV)
        dl_c = torch.zeros(Tc, B, ld, dtype=cdt, device=DEV)
        dl_c[:Ta, :, :V] = dl[:Ta].to(DEV)                              # rows past the step count: zeros (the token pass's contract)
        dh_c = torch.zeros(Tc, B, H, dtype=cdt, device=DEV)
        dh_c[:Ta] = dh[:Ta].to(DEV)
        cap_c = cap.clone()
        cap_c[Ta:] = 0
        grads = [torch.full_like(m, float("nan")) for m in master]
        lo, hid, g_got, df_got = _decoder_call(shape, code, prm, feats, cap_c, dl_c, ld, dh_c, grads, ws, drop, _steps(Ta))
        tol_fwd = 1e-6 if mode == "fp32" else 1e-2                     # the same per-step kernels; the head GEMM's M differs
        assert relerr(hid[:Ta].double().cpu(), hid_ref.double().cpu()) < tol_fwd, Ta
        assert relerr(lo[:Ta].double().cpu(), lo_ref.double().cpu()) < tol_fwd, Ta
        assert torch.equal(hid[Ta:].float().cpu(), torch.zeros(Tc - Ta, B, H)), Ta
        names = ops.param_order(L)
        for name, a, b in zip(names, g_got, g_ref):
            assert torch.isfinite(a).all(), (Ta, name)
            err = relerr(a, b) if mode == "fp32" else relerr_l2(a, b)
            assert err < (1e-5 if mode == "fp32" else 1e-3), (Ta, name, err)
        err = relerr(df_got, df_ref) if mode == "fp32" else relerr_l2(df_got, df_ref)
        assert err < (1e-5 if mode == "fp32" else 1e-3), (Ta, "dfeats", err)


# ------------------------------------------------------------------ 4. graphed step
def _batches(B, V, E, H, lengths, seed):
    out = []
    for i, T in enumerate(lengths):
        b = O.synthetic_batch(B, T, V, E, H, Et=48, seed=seed + i)
        out.append({k: (v.to(DEV) if v is not None else None) for k, v in b.items()})
    return out


def _student(params, pparams, V, E, H, L, mode, dropout=0.0):
    from imagecaptioner_b200.optim import FlatAdamW, reference_param_groups
    model, projector = build_student(params, pparams, V, E, H, L, True, 48, DEV, dropout=dropout)
    if dropout > 0:
        model.train()
    for m in (model.decoder, model.attention_refinement, projector):
        m.compute_dtype = torch.bfloat16 if mode == "bf16" else torch.float32
    # the reference's parameter groups: every group starts on a 16-byte boundary of the flat buffer, so the LayerNorm parameters
    # (read with 16-byte loads) stay aligned although output_projection.3.bias has V = 4999 elements
    return model, projector, FlatAdamW(reference_param_groups(model, projector, 1e-3), weight_decay=0.01, max_grad_norm=1.0)


def _eager_load(kd, batch):
    """Point an eager (use_graph=False, max_steps=None) step at an unpadded batch of its own T."""
    kd.static = {k: batch[k].clone() for k in kd.INPUT_KEYS if batch.get(k) is not None}
    kd.static["encoder_features"].requires_grad_(True)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_graphed_varlen_step_equals_eager_unpadded(mode):
    """GraphedKDStep(max_steps=24), captured once, replayed on batches of T = 24, 9, 17, 1, 24: after every step the loss parts and
    all parameters (FlatAdamW) match a twin model stepped eagerly on the unpadded batches."""
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    V, E, H, L, B = 4999, 64, 128, 2, 64
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(48, E, seed=1)
    batches = _batches(B, V, E, H, [24, 9, 17, 1, 24], seed=40)
    mg, pg, og = _student(params, pparams, V, E, H, L, mode)
    sd0 = og.state_dict()
    kg = GraphedKDStep(mg, pg, DistillationLoss(vocab_size=V), og, None, batches[0], autocast_dtype=None, warmup_steps=1, max_steps=24)
    mg.load_state_dict({k: v.float() for k, v in params.items()}, strict=False)      # undo the warm-up + capture updates
    pg.load_state_dict({k: v.float() for k, v in pparams.items()})
    og.load_state_dict(sd0)
    me, pe, oe = _student(params, pparams, V, E, H, L, mode)
    ke = GraphedKDStep(me, pe, DistillationLoss(vocab_size=V), oe, None, batches[0], autocast_dtype=None, use_graph=False)
    tol_loss, tol_w = (1e-5, 1e-4) if mode == "fp32" else (2e-2, 2e-2)
    for i, b in enumerate(batches):
        kg.load(b)
        lg = kg.step().clone()
        _eager_load(ke, b)
        le = ke.step().clone()
        torch.cuda.synchronize()
        assert torch.isfinite(lg).all(), (i, lg)
        assert relerr(lg.cpu(), le.cpu()) < (tol_loss if i == 0 else tol_w), (i, lg, le)
        err = relerr_l2(og.flat_param.cpu(), oe.flat_param.cpu())
        assert err < tol_w, (i, err)
    with pytest.raises(ValueError):
        kg.load(_batches(B, V, E, H, [25], seed=90)[0])


def test_varlen_dropout_masks_match_unpadded():
    """Dropout p > 0: the masks are counter-based hashes of (seed, site, element index), and the rows of the first T steps have the
    same indices in a (T_cap, B, .) buffer as in a (T, B, .) one, so the variable-length step draws the masks of the unpadded step.
    Compared eagerly (the seed of a captured graph is frozen at capture, so a graph and an eager step never share masks)."""
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    V, E, H, L, B = 4999, 64, 128, 2, 64
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(48, E, seed=1)
    batches = _batches(B, V, E, H, [24, 9, 17], seed=60)
    mv, pv, ov = _student(params, pparams, V, E, H, L, "fp32", dropout=0.3)
    kv = GraphedKDStep(mv, pv, DistillationLoss(vocab_size=V), ov, None, batches[0], autocast_dtype=None, use_graph=False, max_steps=24)
    me, pe, oe = _student(params, pparams, V, E, H, L, "fp32", dropout=0.3)
    ke = GraphedKDStep(me, pe, DistillationLoss(vocab_size=V), oe, None, batches[0], autocast_dtype=None, use_graph=False)
    for i, b in enumerate(batches):
        kv.load(b)
        lv = kv.step().clone()
        _eager_load(ke, b)
        le = ke.step().clone()
        torch.cuda.synchronize()
        assert relerr(lv.cpu(), le.cpu()) < 1e-5, (i, lv, le)
        assert relerr_l2(ov.flat_param.cpu(), oe.flat_param.cpu()) < 1e-4, i


def test_fixed_shape_step_still_rejects_other_lengths():
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    V, E, H, L, B = 200, 32, 64, 1, 8
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(48, E, seed=1)
    b6, b9 = _batches(B, V, E, H, [6, 9], seed=80)
    m, p, o = _student(params, pparams, V, E, H, L, "fp32")
    kd = GraphedKDStep(m, p, DistillationLoss(vocab_size=V), o, None, b6, autocast_dtype=None, use_graph=False)
    assert kd.steps is None and kd.static["captions_input"].shape[0] == 6
    with pytest.raises(RuntimeError):
        kd.load(b9)
    with pytest.raises(ValueError):
        GraphedKDStep(m, p, DistillationLoss(vocab_size=V), o, None, b9, autocast_dtype=None, use_graph=False, max_steps=6)
