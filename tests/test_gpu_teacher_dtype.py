"""GPU: teacher outputs in bf16 / fp16 are read in their own precision (the *_teacher entry points, B2C_BF16 / B2C_F16) and widened
exactly in registers.  Every result must be bit-identical to the same call on `teacher.float()`, or, where atomically added
reductions make two fp32 runs differ, within the spread of two such runs."""
import pytest
import torch

from oracle import kd_oracle as O
from tests.harness import build_student, compare_step, relerr, run_kd_step, to_device

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
HALF = [torch.bfloat16, torch.float16]


def _lib():
    from imagecaptioner_b200 import _ops
    return _ops, _ops.load_library()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _code(ops, dt):
    return {torch.float32: ops.B2C_F32, torch.bfloat16: ops.B2C_BF16, torch.float16: ops.B2C_F16}[dt]


def _at_storage_end(t):
    """`t` copied into a 1-D storage at an odd element offset, as a view that ends exactly where the storage ends."""
    buf = torch.empty(t.numel() + 3, dtype=t.dtype, device=t.device)
    v = buf[3:].view(t.shape)
    v.copy_(t)
    return v


def _token_pass(y, z, tgt, V, ld, cdt, steps=None, B=1, eval_form=False, temp=4.0):
    """One call of b2c_kd_token_loss_teacher (or b2c_kd_token_eval_teacher) -> (rows, dlogits or argmax)."""
    ops, lib = _lib()
    N = tgt.numel()
    nval = ops.count_valid(tgt, V)
    rows = torch.full((2, N), float("nan"), device=DEV)
    if eval_form:
        pred = torch.full((N,), -1, dtype=torch.int32, device=DEV)
        rc = lib.b2c_kd_token_eval_teacher(y.data_ptr(), z.data_ptr(), _code(ops, z.dtype), tgt.data_ptr(), N, V, temp, nval.data_ptr(),
                                           rows[0].data_ptr(), rows[1].data_ptr(), pred.data_ptr(), _code(ops, cdt), _st())
        assert rc == 0, lib.b2c_last_error()
        torch.cuda.synchronize()
        return rows.cpu(), pred.cpu()
    dy = torch.full((N, ld), float("nan"), dtype=cdt, device=DEV)
    rc = lib.b2c_kd_token_loss_teacher(y.data_ptr(), z.data_ptr(), _code(ops, z.dtype), tgt.data_ptr(), N, V, temp, 0.6, 0.25, 1.0,
                                       nval.data_ptr(), dy.data_ptr(), ld, rows[0].data_ptr(), rows[1].data_ptr(), _code(ops, cdt),
                                       None if steps is None else steps.data_ptr(), B, _st())
    assert rc == 0, lib.b2c_last_error()
    torch.cuda.synchronize()
    return rows.cpu(), dy.float().cpu()


def _inputs(V, N, cdt, seed):
    g = torch.Generator().manual_seed(seed)
    y = (torch.randn(N, V, generator=g) * 1.5).to(cdt).to(DEV)
    z = (torch.randn(N, V, generator=g) * 2.5).to(DEV)
    tgt = torch.randint(1, V, (N,), generator=g).to(DEV)
    tgt[::5] = 0
    return y, z, tgt


# ------------------------------------------------------------------ 1. token pass, every form
# (V, student mode, pitch): the aligned pipe, the unaligned pipe with pitched dlogits, the row-in-smem fallback (fp32 mode at
# V = 203, and V > 16384 in both modes)
FORMS = [(5000, "bf16", 5000), (4999, "bf16", 5000), (5001, "bf16", 5008), (203, "fp32", 203), (16400, "fp32", 16400),
         (16400, "bf16", 16400)]


@pytest.mark.parametrize("tdt", HALF)
@pytest.mark.parametrize("V,mode,ld", FORMS)
def test_token_pass_half_teacher_bit_identical(V, mode, ld, tdt):
    cdt = torch.bfloat16 if mode == "bf16" else torch.float32
    N = 96 if V < 10000 else 24
    y, z, tgt = _inputs(V, N, cdt, V)
    zh = z.to(tdt)
    rows_h, dy_h = _token_pass(y, zh, tgt, V, ld, cdt)
    rows_f, dy_f = _token_pass(y, zh.float(), tgt, V, ld, cdt)
    assert torch.equal(rows_h, rows_f)
    assert torch.equal(dy_h, dy_f)
    if V % 8:
        # rows that do not start on a 16-byte boundary and views that end exactly at the end of their storage (guarded first / last rows)
        yv, zv = _at_storage_end(y), _at_storage_end(zh)
        rows_v, dy_v = _token_pass(yv, zv, tgt, V, ld, cdt)
        rows_vf, dy_vf = _token_pass(yv, _at_storage_end(zh.float()), tgt, V, ld, cdt)
        assert torch.equal(rows_v, rows_vf) and torch.equal(dy_v, dy_vf)
        assert torch.equal(rows_v, rows_f) and torch.equal(dy_v, dy_f)


@pytest.mark.parametrize("tdt", HALF)
@pytest.mark.parametrize("V,mode", [(5000, "bf16"), (4999, "bf16"), (203, "fp32")])
def test_token_eval_half_teacher_bit_identical(V, mode, tdt):
    cdt = torch.bfloat16 if mode == "bf16" else torch.float32
    y, z, tgt = _inputs(V, 80, cdt, V + 1)
    zh = z.to(tdt)
    rows_h, pred_h = _token_pass(y, zh, tgt, V, V, cdt, eval_form=True)
    rows_f, pred_f = _token_pass(y, zh.float(), tgt, V, V, cdt, eval_form=True)
    assert torch.equal(rows_h, rows_f) and torch.equal(pred_h, pred_f)


@pytest.mark.parametrize("tdt", HALF)
@pytest.mark.parametrize("V,mode,ld", [(5000, "bf16", 5000), (4999, "bf16", 5000), (203, "fp32", 203)])
def test_token_pass_steps_half_teacher(V, mode, ld, tdt):
    """The step-count form: teacher rows past n = steps * B are NaN and never read; the rest is bit-identical to fp32."""
    cdt = torch.bfloat16 if mode == "bf16" else torch.float32
    Tc, B = 6, 16
    y, z, tgt = _inputs(V, Tc * B, cdt, V + 2)
    for Ta in (1, 4):
        t = tgt.clone()
        t[Ta * B:] = 0
        zh = z.to(tdt)
        zh[Ta * B:] = float("nan")
        steps = torch.full((1,), Ta, dtype=torch.int32, device=DEV)
        rows_h, dy_h = _token_pass(y, zh, t, V, ld, cdt, steps=steps, B=B)
        rows_f, dy_f = _token_pass(y, zh.float(), t, V, ld, cdt, steps=steps, B=B)
        assert torch.equal(rows_h, rows_f) and torch.equal(dy_h, dy_f), Ta
        assert not torch.isnan(dy_h).any() and not torch.isnan(rows_h).any()


# ------------------------------------------------------------------ 2. hidden KD
@pytest.mark.parametrize("tdt", HALF)
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_aux_loss_half_teacher_hiddens(mode, tdt):
    ops, lib = _lib()
    Tc, B, H, E, Ss, St = 6, 8, 64, 32, 10, 12
    cdt = torch.bfloat16 if mode == "bf16" else torch.float32
    code = _code(ops, cdt)
    g = torch.Generator().manual_seed(3)
    fs = torch.randn(B, Ss, E, generator=g).to(DEV)
    ft = torch.randn(B, St, E, generator=g).to(DEV)
    hs = torch.randn(Tc, B, H, generator=g).to(cdt).to(DEV)
    ht = torch.randn(Tc, B, H, generator=g).to(tdt).to(DEV)

    def run(ht_, steps):
        dfs, dft = torch.empty(B, Ss, E, device=DEV), torch.empty(B, St, E, device=DEV)
        dhs = torch.full((Tc, B, H), float("nan"), dtype=cdt, device=DEV)
        fp, hp = torch.empty(B, 2, device=DEV), torch.full((Tc * B, 2), float("nan"), device=DEV)
        rc = lib.b2c_aux_loss_teacher(fs.data_ptr(), ft.data_ptr(), B, Ss, St, E, hs.data_ptr(), ht_.data_ptr(), _code(ops, ht_.dtype), Tc, Tc,
                                      H, 0.2, 0.1, dfs.data_ptr(), dft.data_ptr(), dhs.data_ptr(), fp.data_ptr(), hp.data_ptr(), code,
                                      ops.B2C_F32, None if steps is None else steps.data_ptr(), _st())
        assert rc == 0, lib.b2c_last_error()
        torch.cuda.synchronize()
        return [t.float().cpu() for t in (hp, dhs, fp, dfs, dft)]

    for steps in (None, torch.full((1,), 4, dtype=torch.int32, device=DEV)):
        a, b = run(ht, steps), run(ht.float(), steps)
        for x, y in zip(a, b):
            assert torch.equal(x, y)


# ------------------------------------------------------------------ 3. projector
@pytest.mark.parametrize("tdt", HALF)
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("learned", [True, False])
def test_projector_half_teacher_features(learned, mode, tdt):
    from imagecaptioner_b200.distillation_utils import FeatureProjector
    Et, Es, B = (48, 64, 6) if learned else (64, 64, 6)
    proj = FeatureProjector(Et, Es, 197, 49).to(DEV).eval()
    proj.compute_dtype = torch.bfloat16 if mode == "bf16" else torch.float32
    g = torch.Generator().manual_seed(9)
    x = torch.randn(B, 197, Et, generator=g).to(tdt).to(DEV)
    dout = torch.randn(B, 49, Es, generator=g).to(DEV)

    def run(inp):
        proj.zero_grad(set_to_none=True)
        out = proj(inp)
        if learned:
            (out * dout).sum().backward()
        torch.cuda.synchronize()
        return out.detach().cpu(), [p.grad.detach().cpu() for p in proj.parameters() if p.grad is not None]

    out_h, g_h = run(x)
    out_a, g_a = run(x.float())
    out_b, g_b = run(x.float())
    assert torch.equal(out_h, out_a)
    for gh, ga, gb in zip(g_h, g_a, g_b):
        spread = relerr(gb, ga)
        assert relerr(gh, ga) <= max(2 * spread, 1e-6), (relerr(gh, ga), spread)


# ------------------------------------------------------------------ 4. fused validation
@pytest.mark.parametrize("tdt", HALF)
@pytest.mark.parametrize("V", [5000, 4999])
def test_fused_validation_half_teacher(V, tdt):
    from imagecaptioner_b200 import _ops
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    B, T, E, H, L, Et = 24, 5, 64, 128, 2, 48
    params = O.init_student_params(V, E, H, L, True, seed=31, logit_scale=6.0)
    pparams = O.init_projector_params(Et, E, seed=32)
    batch = O.synthetic_batch(B, T, V, E, H, Et=Et, seed=33)
    model, projector = build_student(params, pparams, V, E, H, L, True, Et, DEV)
    for m in (model.decoder, model.attention_refinement, projector):
        m.compute_dtype = torch.bfloat16
    loss_mod = DistillationLoss(0.5, 0.2, 0.1, 4.0, vocab_size=V)
    d = to_device(batch, DEV)
    zh = d["teacher_logits"].to(tdt)
    hid_t = d["teacher_hiddens"].to(tdt)
    res = []
    with torch.no_grad():
        for z, ht, ft in ((zh, hid_t, d["teacher_features"].to(tdt)), (zh.float(), hid_t.float(), d["teacher_features"].to(tdt).float())):
            rows, pred, _, _, _ = model.forward_validation(d["encoder_features"], d["captions_input"], z, d["targets"], 4.0)
            t_out = {"logits": z, "encoder_features": projector(ft), "hidden_states": ht}
            _, parts, pred_f = loss_mod.evaluate_fused(model, d["encoder_features"], d["captions_input"], t_out, d["targets"])
            logits, enc, hids, _ = model(d["encoder_features"], d["captions_input"])
            _, parts_u, pred_u = loss_mod.evaluate({"logits": logits, "encoder_features": enc, "hidden_states": hids}, t_out, d["targets"])
            torch.cuda.synchronize()
            res.append((rows.cpu(), pred.cpu(), _ops.bleu1(pred, d["targets"]).cpu(), parts, pred_f.cpu(), parts_u, pred_u.cpu()))
    for a, b in zip(*res):
        if isinstance(a, dict):
            assert a == b
        else:
            assert torch.equal(a, b)


# ------------------------------------------------------------------ 5. DistillationLoss with fp16 teacher outputs
def test_distillation_loss_config1_fp16_teacher_matches_oracle():
    """BASELINE config 1 shapes with the teacher's logits, features and hidden states in fp16: the fp32 step agrees with the fp64
    oracle on the upcast values at the fp32 parity tolerance."""
    m = dict(B=16, T=20, V=5000, E=256, H=512, L=2)
    params = O.init_student_params(m["V"], m["E"], m["H"], m["L"], True, seed=0)
    pparams = O.init_projector_params(384, m["E"], seed=1)
    batch = O.synthetic_batch(m["B"], m["T"], m["V"], m["E"], m["H"], seed=2)
    half = dict(batch)
    for k in ("teacher_logits", "teacher_features", "teacher_hiddens"):
        half[k] = batch[k].to(torch.float16)
    up = dict(half)
    for k in ("teacher_logits", "teacher_features", "teacher_hiddens"):
        up[k] = half[k].double()
    ref = O.kd_step(to_device(params, DEV), to_device(pparams, DEV), to_device(up, DEV), dtype=torch.float64)
    ref = {k: ({kk: (vv.cpu() if torch.is_tensor(vv) else vv) for kk, vv in v.items()} if isinstance(v, dict) else v.cpu()) for k, v in ref.items()}
    model, projector = build_student(params, pparams, m["V"], m["E"], m["H"], m["L"], True, 384, DEV)
    got = run_kd_step(model, projector, half, DEV, torch.float32)
    compare_step(got, ref, 2e-4, verbose=False)


def test_distillation_loss_half_teacher_makes_no_fp32_copy():
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    T, B, V = 20, 64, 5000
    g = torch.Generator().manual_seed(4)
    y = (torch.randn(T, B, V, generator=g)).to(torch.bfloat16).to(DEV).requires_grad_(True)
    z = (torch.randn(T, B, V, generator=g) * 2).to(torch.float16).to(DEV)
    tgt = torch.randint(1, V, (T, B), generator=g).to(DEV)
    loss_mod = DistillationLoss(vocab_size=V)
    loss_mod({"logits": y}, {"logits": z}, tgt)          # warm-up: library load, kernel attributes
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    total, parts = loss_mod({"logits": y}, {"logits": z}, tgt)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown < z.numel() * 4, (grown, z.numel() * 4)
    _, parts_f = loss_mod({"logits": y}, {"logits": z.float()}, tgt)
    assert parts == parts_f


# ------------------------------------------------------------------ 6. graphed step
@pytest.mark.parametrize("max_steps", [None, 8])
def test_graphed_step_bf16_teacher(max_steps):
    from imagecaptioner_b200.ddp import FlatGradAllReducer
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    V, E, H, L, B, T = 5000, 64, 128, 2, 8, 6
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(48, E, seed=1)
    b32 = {k: v for k, v in O.synthetic_batch(B, T, V, E, H, Et=48, seed=7).items() if v is not None}
    teacher_keys = ("teacher_logits", "teacher_features", "teacher_hiddens")
    b16 = {k: (v.to(torch.bfloat16) if k in teacher_keys else v) for k, v in b32.items()}
    bup = {k: (v.float() if k in teacher_keys else v) for k, v in b16.items()}
    out, weights, loaded = [], [], []
    for batch in (b16, bup):
        model, projector = build_student(params, pparams, V, E, H, L, True, 48, DEV)
        for m in (model.decoder, model.attention_refinement, projector):
            m.compute_dtype = torch.bfloat16
        trainable = [p for p in list(model.parameters()) + list(projector.parameters()) if p.requires_grad]
        opt = torch.optim.AdamW(trainable, lr=1e-3, weight_decay=0.01, fused=True, capturable=True)
        dev_batch = {k: v.to(DEV) for k, v in batch.items()}
        kd = GraphedKDStep(model, projector, DistillationLoss(vocab_size=V), opt, FlatGradAllReducer(trainable), dev_batch,
                           autocast_dtype=None, warmup_steps=1, max_steps=max_steps)
        model.load_state_dict({k: v.float() for k, v in params.items()}, strict=False)      # undo the warm-up step's update
        projector.load_state_dict({k: v.float() for k, v in pparams.items()})
        host = {k: v.pin_memory() for k, v in batch.items()}
        steps = []
        for _ in range(3):
            loaded.append(kd.load(host))
            steps.append(kd.step().clone())
        torch.cuda.synchronize()
        out.append(torch.stack(steps).cpu())
        weights.append(torch.cat([p.detach().float().flatten() for p in trainable]).cpu())
    assert relerr(out[0][0], out[1][0]) < 1e-6
    assert relerr(out[0], out[1]) < 2e-2
    assert relerr(weights[0], weights[1]) < 2e-2
    teacher_bytes = sum(b32[k].numel() * 4 for k in teacher_keys)
    assert loaded[3] - loaded[0] == teacher_bytes // 2


def test_graphed_step_half_teacher_launches_no_cast():
    """One step with bf16 teacher tensors launches exactly the non-native kernels of the step with fp32 teacher tensors: no
    conversion of the teacher tensors (the captured graph records the same launches)."""
    from torch.profiler import ProfilerActivity, profile
    from imagecaptioner_b200.ddp import FlatGradAllReducer
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    V, E, H, L, B, T = 5000, 64, 128, 2, 8, 6
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(48, E, seed=1)
    b32 = {k: v.to(DEV) for k, v in O.synthetic_batch(B, T, V, E, H, Et=48, seed=7).items() if v is not None}
    b16 = {k: (v.to(torch.bfloat16) if k.startswith("teacher_") else v) for k, v in b32.items()}
    counts = []
    for batch in (b32, b16):
        model, projector = build_student(params, pparams, V, E, H, L, True, 48, DEV)
        for m in (model.decoder, model.attention_refinement, projector):
            m.compute_dtype = torch.bfloat16
        trainable = [p for p in list(model.parameters()) + list(projector.parameters()) if p.requires_grad]
        opt = torch.optim.AdamW(trainable, lr=1e-3, weight_decay=0.01, fused=True, capturable=True)
        kd = GraphedKDStep(model, projector, DistillationLoss(vocab_size=V), opt, FlatGradAllReducer(trainable), batch,
                           autocast_dtype=None, use_graph=False)
        kd.step()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            kd.step()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        counts.append(sum(1 for n in names if "b2c" not in n))
    assert counts[0] == counts[1], counts


# ------------------------------------------------------------------ 7. errors
def test_unknown_teacher_dtype_and_float64_teacher():
    ops, lib = _lib()
    V, N = 64, 16
    y, z, tgt = _inputs(V, N, torch.float32, 5)
    nval = ops.count_valid(tgt, V)
    rows = torch.empty(2, N, device=DEV)
    dy = torch.empty(N, V, device=DEV)
    rc = lib.b2c_kd_token_loss_teacher(y.data_ptr(), z.data_ptr(), 7, tgt.data_ptr(), N, V, 4.0, 0.6, 0.25, 1.0, nval.data_ptr(),
                                       dy.data_ptr(), V, rows[0].data_ptr(), rows[1].data_ptr(), ops.B2C_F32, None, 1, _st())
    assert rc == -1 and b"teacher dtype" in lib.b2c_last_error()
    rc = lib.b2c_kd_token_eval(y.data_ptr(), z.data_ptr(), tgt.data_ptr(), N, V, 4.0, nval.data_ptr(), rows[0].data_ptr(),
                               rows[1].data_ptr(), None, ops.B2C_F16, _st())
    assert rc == -1                                        # B2C_F16 is a teacher dtype only, never a compute dtype
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    loss_mod = DistillationLoss(vocab_size=V)
    yl = y.view(4, 4, V)
    _, p64 = loss_mod({"logits": yl}, {"logits": z.view(4, 4, V).double()}, tgt.view(4, 4))
    _, p32 = loss_mod({"logits": yl}, {"logits": z.view(4, 4, V)}, tgt.view(4, 4))
    assert p64 == p32
