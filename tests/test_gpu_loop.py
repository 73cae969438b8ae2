"""GPU: the reference's OWN call pattern around the hot path, replayed on the drop-in modules.

`train_student_kd.py` / `evaluate_student.py` cannot be imported here or on the GPU box (timm, spaCy, Flickr8k, a teacher checkpoint,
hard-coded paths), so this test replays the structure of their training-loop body statement by statement
(/root/reference/src/train_student_kd.py:202-303): validate_distillation_setup -> create_feature_projectors, TeacherWrapper, three-group
stock AdamW, fp16 `autocast('cuda')`, `GradScaler('cuda')`, `loss / accumulation_steps`, `scaler.scale(loss).backward()`, and every second
batch `unscale_`, `clip_grad_norm_` on the student and on EVERY projector, `scaler.step`, `scaler.update`, `zero_grad`, `scheduler.step`.
The same loop on the CPU oracle (fp32) is the reference."""
import math

import pytest
import torch
import torch.nn as nn

from oracle import kd_oracle as O
from tests.harness import build_student, relerr, relerr_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
V, E, H, L, B, T, ET_DIM = 200, 64, 128, 2, 8, 6, 48


class StubTeacher(nn.Module):
    """What TeacherWrapper touches (/root/reference/src/distillation_utils.py:268-292): teacher(images, captions) -> logits,
    teacher.encoder.forward_features(images) -> ViT tokens, teacher.encoder_projection(tokens); plus the attributes
    create_feature_projectors reads (:295-340).  It replays a fixed list of synthetic batches."""

    class _Enc(nn.Module):
        def __init__(self, outer):
            super().__init__()
            self._outer = [outer]
            self.num_features = ET_DIM

        def forward_features(self, images):
            o = self._outer[0]
            return o.batches[o.cursor]["teacher_features"].to(images.device)

    def __init__(self, batches):
        super().__init__()
        self.batches, self.cursor = batches, 0
        self.encoder = self._Enc(self)
        self.encoder_projection = nn.Identity()          # no out_features / in_features: the projector dim falls back to encoder.num_features
        self.embed_size = H + 16                         # 'hidden' projector Linear(H+16 -> H): has parameters, is never called in the loop
        self.dummy = nn.Parameter(torch.zeros(1))

    def forward(self, images, captions):
        return self.batches[self.cursor]["teacher_logits"].to(images.device)


def _batches(n):
    return [O.synthetic_batch(B, T, V, E, H, Et=ET_DIM, seed=100 + i, teacher_hiddens=False) for i in range(n)]


def _captions(b):                                        # (T+1, B): input = [:-1], target = [1:]  (:262-263)
    return torch.cat([b["captions_input"], b["targets"][-1:]], dim=0)


def _run_reference_loop(student, teacher, batches, autocast_on, lr=2e-3, accumulation_steps=2):
    from imagecaptioner_b200.distillation_utils import DistillationLoss, TeacherWrapper, validate_distillation_setup
    from torch.amp import GradScaler, autocast
    from torch.optim.lr_scheduler import CosineAnnealingWarmRestarts
    device = torch.device(DEV)
    # :202  (dry run with the UNSHIFTED captions as targets, outside autocast, grad enabled)
    teacher.cursor = 0
    sample = (batches[0]["encoder_features"].to(device), batches[0]["captions_input"].to(device))
    projectors, distill_loss = validate_distillation_setup(teacher, student, sample)
    assert set(projectors) == {"encoder", "hidden"} and tuple(projectors["encoder"](batches[0]["teacher_features"].to(device)).shape) == (B, 49, E)
    for pr in projectors.values():
        pr.eval()                                        # parity needs dropout off (the reference's loop runs train(): p = 0.3 / 0.1)
    # the stub's projector weights are random per construction: pin them so the oracle can use the same ones
    pparams = O.init_projector_params(ET_DIM, E, seed=1)
    projectors["encoder"].load_state_dict({k: v.float() for k, v in pparams.items()})
    projectors["encoder"].to(device)
    distill_loss = DistillationLoss(alpha=0.7, beta=0.2, gamma=0.1, temperature=4.0, vocab_size=V)       # :205-211
    encoder_params = list(student.encoder.parameters())                                                   # :219-234
    decoder_params = list(student.decoder.parameters())
    other_params = list(student.attention_refinement.parameters())
    for projector in projectors.values():
        other_params.extend(list(projector.parameters()))
    groups = [{"params": decoder_params, "lr": lr}, {"params": other_params, "lr": lr}]
    if encoder_params:
        groups.insert(0, {"params": encoder_params, "lr": lr * 0.1})
    optimizer = torch.optim.AdamW(groups, weight_decay=0.01)
    scheduler = CosineAnnealingWarmRestarts(optimizer, T_0=5, T_mult=2, eta_min=1e-6)                    # :236
    scaler = GradScaler("cuda", enabled=autocast_on)                                                      # :239
    teacher_wrapper = TeacherWrapper(teacher)
    losses = []
    for batch_idx, b in enumerate(batches):                                                               # :258-303
        teacher.cursor = batch_idx
        imgs, captions = b["encoder_features"].to(device), _captions(b).to(device)
        captions_input, captions_target = captions[:-1, :], captions[1:, :]
        teacher_outputs = teacher_wrapper(imgs.float(), captions_input.long())
        with autocast("cuda", enabled=autocast_on):
            logits, enc_feats, hidden_states, _ = student(imgs, captions_input)
            student_outputs = {"logits": logits, "encoder_features": enc_feats, "hidden_states": hidden_states}
            teacher_outputs["encoder_features"] = projectors["encoder"](teacher_outputs["encoder_features"])
            loss, loss_dict = distill_loss(student_outputs, teacher_outputs, captions_target)
            loss = loss / accumulation_steps
        scaler.scale(loss).backward()
        if (batch_idx + 1) % accumulation_steps == 0:
            scaler.unscale_(optimizer)
            torch.nn.utils.clip_grad_norm_(student.parameters(), max_norm=1.0)
            for projector in projectors.values():
                torch.nn.utils.clip_grad_norm_(projector.parameters(), max_norm=1.0)
            scaler.step(optimizer)
            scaler.update()
            optimizer.zero_grad()
            scheduler.step(0 + batch_idx / len(batches))
        losses.append(loss.item() * accumulation_steps)
        assert set(loss_dict) == {"total_loss", "ce_loss", "token_kd_loss", "feature_kd_loss", "hidden_kd_loss"} and loss_dict["hidden_kd_loss"] == 0.0
    weights = {k: v.detach().float().cpu().clone() for k, v in student.state_dict().items()}
    weights.update({"proj." + k: v.detach().float().cpu().clone() for k, v in projectors["encoder"].state_dict().items()})
    return losses, weights, float(scaler.get_scale()) if autocast_on else None, projectors


def _oracle_loop(params, pparams, batches, lr=2e-3, accumulation_steps=2):
    from torch.optim.lr_scheduler import CosineAnnealingWarmRestarts
    P = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    Q = {k: v.clone().requires_grad_(True) for k, v in pparams.items()}
    dec = [v for k, v in P.items() if k.startswith("decoder.")]
    other = [v for k, v in P.items() if not k.startswith("decoder.")] + list(Q.values())
    opt = torch.optim.AdamW([{"params": dec, "lr": lr}, {"params": other, "lr": lr}], weight_decay=0.01)
    sched = CosineAnnealingWarmRestarts(opt, T_0=5, T_mult=2, eta_min=1e-6)
    losses = []
    for i, b in enumerate(batches):
        out, enc, hids, _ = O.student_forward(P, b["encoder_features"], b["captions_input"], True)
        tproj = O.feature_projector(Q, b["teacher_features"], 49)
        total, _ = O.distillation_loss({"logits": out, "encoder_features": enc, "hidden_states": hids},
                                       {"logits": b["teacher_logits"], "encoder_features": tproj, "hidden_states": None}, b["targets"])
        (total / accumulation_steps).backward()
        if (i + 1) % accumulation_steps == 0:
            torch.nn.utils.clip_grad_norm_(list(P.values()), 1.0)
            torch.nn.utils.clip_grad_norm_(list(Q.values()), 1.0)
            opt.step(); opt.zero_grad(); sched.step(0 + i / len(batches))
        losses.append(float(total.detach()))
    w = {k: v.detach().clone() for k, v in P.items()}
    w.update({"proj." + k: v.detach().clone() for k, v in Q.items()})
    return losses, w


@pytest.mark.parametrize("autocast_on", [False, True])
def test_reference_training_loop_replay(autocast_on):
    """4 batches, accumulation_steps = 2 (two optimizer steps).  fp32 (autocast off): losses and updated weights equal the CPU oracle
    loop.  fp16-autocast + GradScaler (the reference's real configuration; the native modules run their bf16 mode under autocast, a
    2^15-scaled grad_output goes through b2c_scale_inplace): losses within the bf16 tolerance, the loss scale is intact (no inf / nan
    skipped a step), and the weight UPDATE points the same way as the oracle's."""
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(ET_DIM, E, seed=1)
    batches = _batches(4)
    ref_losses, ref_w = _oracle_loop(params, pparams, batches)
    student, _ = build_student(params, pparams, V, E, H, L, True, ET_DIM, DEV)
    losses, w, scale, projectors = _run_reference_loop(student, StubTeacher(batches), batches, autocast_on)
    init = dict(params); init.update({"proj." + k: v for k, v in pparams.items()})
    tol = 2e-2 if autocast_on else 1e-4
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= tol * abs(b), (losses, ref_losses)
    # the 'hidden' projector never receives a gradient: stock AdamW leaves it untouched (no weight decay either)
    hp = projectors["hidden"]
    assert len(list(hp.parameters())) == 4 and all(p.grad is None for p in hp.parameters())
    worst = 0.0
    for k, v in ref_w.items():
        du_ref, du = (v - init[k]).double(), (w[k] - init[k].float()).double()
        if float(du_ref.abs().max()) == 0.0:
            assert float(du.abs().max()) == 0.0, k
            continue
        if autocast_on:
            cos = float((du * du_ref).sum() / (du.norm() * du_ref.norm() + 1e-30))
            assert cos > 0.9, (k, cos)                   # Adam normalises every element to +-lr: bf16 noise flips near-zero gradients only
        else:
            # Adam maps a ~1e-9 gradient to a +-lr step, so single elements may differ between two summation orders: L2 over the tensor
            # Adam maps a gradient below eps = 1e-8 to a partial step (slope 1/eps), so the rare elements whose gradient is ~0 amplify
            # fp32 round-off: the update is compared in L2 over the tensor (2e-2) and in the max norm with room for those elements;
            # a wrong clip group, accumulation factor or loss-scale handling is an O(1) error in both
            worst = max(worst, relerr_l2(du, du_ref))
            assert relerr_l2(du, du_ref) < 2e-2, k
            assert relerr(du, du_ref) < 0.6, k
    if autocast_on:
        assert scale == 65536.0                          # GradScaler's initial scale: no step was skipped, no inf / nan in the gradients
    assert all(math.isfinite(x) for x in losses)


def test_eager_accumulation_after_graphed_step_is_not_redirected():
    """A GraphedKDStep writes gradients straight into its flat buffer (overwrite semantics).  Those destinations are per-call
    options attached only inside its own step, so an eager loop on the same model afterwards ACCUMULATES like autograd does
    (ADVICE round 1: a process-global destination table broke accumulation_steps > 1)."""
    from imagecaptioner_b200.distillation_utils import DistillationLoss
    from imagecaptioner_b200.graph import GraphedKDStep
    from imagecaptioner_b200.optim import FlatAdamW, reference_param_groups
    from tests.harness import run_kd_step
    params = O.init_student_params(V, E, H, L, True, seed=0)
    pparams = O.init_projector_params(ET_DIM, E, seed=1)
    batch = O.synthetic_batch(B, T, V, E, H, Et=ET_DIM, seed=7)
    dev_batch = {k: (v.to(DEV) if v is not None else None) for k, v in batch.items()}
    model, projector = build_student(params, pparams, V, E, H, L, True, ET_DIM, DEV)
    model.decoder.compute_dtype = torch.float32
    opt = FlatAdamW(reference_param_groups(model, projector, 0.0), weight_decay=0.0, max_grad_norm=1.0)      # lr 0: weights stay put
    kd = GraphedKDStep(model, projector, DistillationLoss(vocab_size=V), opt, None, dev_batch, autocast_dtype=None, warmup_steps=1)
    kd.step(); torch.cuda.synchronize()
    assert getattr(model.decoder, "b2c_options", None) is None
    g1 = run_kd_step(model, projector, batch, DEV, torch.float32)["grads"]["decoder.lstm.weight_hh_l0"]
    # second backward WITHOUT zeroing: .grad must now hold twice the gradient
    feats = dev_batch["encoder_features"].clone().requires_grad_(True)
    out, enc, hids, _ = model(feats, dev_batch["captions_input"])
    tp = projector(dev_batch["teacher_features"])
    th = dev_batch["teacher_hiddens"]
    loss, _ = DistillationLoss(vocab_size=V)({"logits": out, "encoder_features": enc, "hidden_states": hids},
                                             {"logits": dev_batch["teacher_logits"], "encoder_features": tp,
                                              "hidden_states": [th[t] for t in range(th.shape[0])]}, dev_batch["targets"])
    loss.backward()
    g2 = model.decoder.lstm.weight_hh_l0.grad.detach().float().cpu()
    assert relerr(g2, 2 * g1) < 1e-5


def test_two_rank_nccl_step_equals_global_batch(tmp_path):
    """bench.py --check under torchrun on 2 GPUs (NCCL): the averaged all-reduced gradient, the loss parts and the weights after 3
    optimizer steps equal a 1-GPU run on the concatenated batch, with the overlapped exchange and with serial collectives.
    Skipped on a one-GPU box (there, the same control flow runs with identity collectives in test_graphed_step_equals_eager_step
    and `bench.py --check`); profiles/r2_check_dp_n2.json holds the 2-GPU result of this round."""
    import json
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path / "check_n2_test.json")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", os.path.join(root, "bench.py"), "--gpus", "2", "--check", "--out", out],
                       cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    rep = json.load(open(out))
    assert rep["ok"] and rep["overlap_comm_1"]["overlapped_exchange"] and rep["overlap_comm_1"]["grad_step1_rel_err_worst_tensor"] < 1e-4
