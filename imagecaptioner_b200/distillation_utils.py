"""Drop-in for the reference's ``src/distillation_utils.py`` (the loss API of the KD hot path).

Same public names, constructor arguments, dict keys and error behaviour as
``/root/reference/src/distillation_utils.py``; ``DistillationLoss.forward`` is two fused sm_100a
kernels (the streaming token KD + CE pass producing loss and dlogits, and the feature/hidden KD
reduction) plus a fixed-order finalize, instead of ~40 eager launches and 5 host syncs.
``FeatureProjector`` keeps its parameters in the reference's stock submodules and computes through
``b2c_projector_forward`` / ``_backward`` (SURVEY.md §8f row 2);
``TeacherWrapper`` / ``create_feature_projectors`` / ``validate_distillation_setup`` /
``compute_bleu_score`` / ``log_training_progress`` are host-side glue with the reference's behaviour.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch
import torch.nn as nn

from . import _ops


def _stack_hidden(states) -> Optional[torch.Tensor]:
    """list of T (B,H) tensors -> (T,B,H); free when the list came from our decoder."""
    if states is None:
        return None
    if isinstance(states, torch.Tensor):
        return states
    base = getattr(states, "stacked", None)
    if base is not None and base.shape[0] == len(states):
        return base
    return torch.stack(list(states), dim=0)


class DistillationLoss(nn.Module):
    """(1-a-b-g)*CE(ignore PAD) + a*T^2*KL + b*featureKD + g*hiddenKD   (reference :8-200)."""

    def __init__(self, alpha=0.7, beta=0.2, gamma=0.1, temperature=4.0, vocab_size=None):
        super().__init__()
        self.alpha = alpha
        self.beta = beta
        self.gamma = gamma
        self.temperature = temperature
        self.vocab_size = vocab_size
        # data parallelism: set by imagecaptioner_b200.ddp so CE divides by the GLOBAL non-PAD count
        self.process_group = None
        self.world_size = 1
        # optional int32 device scalar holding the (global) non-PAD target count, set by a caller that computes it
        # itself (GraphedKDStep keeps the NCCL all-reduce of the count outside its CUDA graphs)
        self.n_valid_global = None
        # set by a caller that runs `loss.backward()` itself with grad_output == 1 (GraphedKDStep): skips the rescaling pass
        self.assume_unit_grad = False

    # ---- the fused path -------------------------------------------------------------------------
    def _run(self, logits, teacher_logits, targets, feats_s, feats_t, hid_s, hid_t, alpha, beta, gamma, w_ce, temperature):
        if feats_s is not None and feats_t is not None and feats_s.shape[-1] != feats_t.shape[-1]:
            raise ValueError(f"Feature dimensions don't match: student {feats_s.shape[-1]}, teacher {feats_t.shape[-1]}")
        if hid_s is not None and hid_t is not None:
            if hid_s.shape[-1] != hid_t.shape[-1]:
                raise ValueError(f"Hidden dimensions don't match: student {hid_s.shape[-1]}, teacher {hid_t.shape[-1]}")
            n = min(hid_s.shape[0], hid_t.shape[0])           # the reference truncates both lists (:111-113)
            hid_t = hid_t[:n]
        else:
            hid_s = hid_t = None
        if feats_s is None or feats_t is None:
            feats_s = feats_t = None
        opts = getattr(self, "b2c_options", None)           # GraphedKDStep(max_steps=...): the variable-length batch's step count
        cfg = (alpha, beta, gamma, temperature, w_ce, float(self.world_size), self.process_group, self.n_valid_global, self.assume_unit_grad,
               getattr(opts, "steps_dev", None))
        return _ops.KDLossFunction.apply(logits, teacher_logits, targets, feats_s, feats_t, hid_s, hid_t, cfg)

    def forward_device(self, student_outputs, teacher_outputs, targets):
        """Like forward() but with no host sync: returns (loss, out5) where out5 is the device tensor
        [total, ce, token_kd, feature_kd, hidden_kd]."""
        s_logits = student_outputs["logits"]
        t_logits = teacher_outputs["logits"]
        feats_s = feats_t = hid_s = hid_t = None
        if "encoder_features" in student_outputs and "encoder_features" in teacher_outputs:
            feats_s, feats_t = student_outputs["encoder_features"], teacher_outputs["encoder_features"]
        if "hidden_states" in student_outputs and "hidden_states" in teacher_outputs:
            hid_s, hid_t = _stack_hidden(student_outputs["hidden_states"]), _stack_hidden(teacher_outputs["hidden_states"])
        w_ce = 1 - self.alpha - self.beta - self.gamma                # 2.8e-17 at the defaults, honoured as is
        return self._run(s_logits, t_logits, targets, feats_s, feats_t, hid_s, hid_t,
                         self.alpha, self.beta, self.gamma, w_ce, self.temperature)

    def forward(self, student_outputs, teacher_outputs, targets):
        """-> (total_loss 0-dim tensor with grad, loss_dict of 5 Python floats); ONE device->host copy."""
        loss, out5 = self.forward_device(student_outputs, teacher_outputs, targets)
        vals = out5.tolist()
        loss_dict = {"total_loss": vals[0], "ce_loss": vals[1], "token_kd_loss": vals[2],
                     "feature_kd_loss": vals[3], "hidden_kd_loss": vals[4]}
        return loss, loss_dict

    @torch.no_grad()
    def evaluate(self, student_outputs, teacher_outputs, targets):
        """Validation form (reference src/train_student_kd.py:56-75): the same loss WITHOUT gradients, and the teacher-forced
        predictions ``student_logits.argmax(dim=-1)`` from the same pass over the logits.
        -> (total_loss 0-dim tensor, loss_dict of 5 floats, predicted_tokens (T,B) int32 on the device)."""
        feats_s = feats_t = hid_s = hid_t = None
        if "encoder_features" in student_outputs and "encoder_features" in teacher_outputs:
            feats_s, feats_t = student_outputs["encoder_features"], teacher_outputs["encoder_features"]
            if feats_s is not None and feats_t is not None and feats_s.shape[-1] != feats_t.shape[-1]:
                raise ValueError(f"Feature dimensions don't match: student {feats_s.shape[-1]}, teacher {feats_t.shape[-1]}")
        if "hidden_states" in student_outputs and "hidden_states" in teacher_outputs:
            hid_s, hid_t = _stack_hidden(student_outputs["hidden_states"]), _stack_hidden(teacher_outputs["hidden_states"])
            if hid_s is not None and hid_t is not None:
                if hid_s.shape[-1] != hid_t.shape[-1]:
                    raise ValueError(f"Hidden dimensions don't match: student {hid_s.shape[-1]}, teacher {hid_t.shape[-1]}")
                hid_t = hid_t[:min(hid_s.shape[0], hid_t.shape[0])]
            else:
                hid_s = hid_t = None
        w_ce = 1 - self.alpha - self.beta - self.gamma
        out5, pred = _ops.kd_eval(student_outputs["logits"], teacher_outputs["logits"], targets, feats_s, feats_t, hid_s, hid_t,
                                  self.alpha, self.beta, self.gamma, self.temperature, w_ce, self.n_valid_global, float(self.world_size))
        vals = out5.tolist()
        loss_dict = {"total_loss": vals[0], "ce_loss": vals[1], "token_kd_loss": vals[2],
                     "feature_kd_loss": vals[3], "hidden_kd_loss": vals[4]}
        return out5[0], loss_dict, pred

    @torch.no_grad()
    def evaluate_fused(self, student_model, images, captions_input, teacher_outputs, targets):
        """`evaluate` without a logits tensor: the student's validation forward reduces the vocabulary head straight to the per-row
        token-KD / CE partials and the argmax (CaptioningStudent.forward_validation); the feature / hidden terms and the weighting
        follow as in `evaluate`.  -> (total_loss 0-dim tensor, loss_dict of 5 floats, predicted_tokens (T,B) int32)."""
        rows, pred, enc, hids, _ = student_model.forward_validation(images, captions_input, teacher_outputs["logits"], targets, self.temperature)
        feats_t = teacher_outputs.get("encoder_features")
        feats_s = enc if feats_t is not None else None
        if feats_s is not None and feats_s.shape[-1] != feats_t.shape[-1]:
            raise ValueError(f"Feature dimensions don't match: student {feats_s.shape[-1]}, teacher {feats_t.shape[-1]}")
        hid_s, hid_t = _stack_hidden(hids), _stack_hidden(teacher_outputs.get("hidden_states"))
        if hid_t is not None:
            if hid_s.shape[-1] != hid_t.shape[-1]:
                raise ValueError(f"Hidden dimensions don't match: student {hid_s.shape[-1]}, teacher {hid_t.shape[-1]}")
            hid_t = hid_t[:min(hid_s.shape[0], hid_t.shape[0])]
        else:
            hid_s = None
        w_ce = 1 - self.alpha - self.beta - self.gamma
        out5, pred = _ops.kd_eval_rows(rows, pred, targets, student_model.vocab_size, feats_s, feats_t, hid_s, hid_t, self.alpha, self.beta,
                                       self.gamma, self.temperature, w_ce, self.n_valid_global, float(self.world_size))
        vals = out5.tolist()
        loss_dict = {"total_loss": vals[0], "ce_loss": vals[1], "token_kd_loss": vals[2],
                     "feature_kd_loss": vals[3], "hidden_kd_loss": vals[4]}
        return out5[0], loss_dict, pred

    # ---- the reference's individual terms, each through the same kernels --------------------------
    def _dummy_targets(self, logits):
        # any non-PAD id: the CE term is weighted by exactly 0 in the single-term entry points below
        return torch.ones(logits.shape[:-1], dtype=torch.int64, device=logits.device)

    def token_level_distillation(self, student_logits, teacher_logits, temperature=None):
        """T^2 * KL(softmax(teacher/T) || softmax(student/T)), batchmean over all rows (reference :30-54)."""
        temperature = self.temperature if temperature is None else temperature
        V = student_logits.shape[-1]
        y = student_logits.reshape(1, -1, V)
        z = teacher_logits.reshape(1, -1, V)
        loss, _ = self._run(y, z, self._dummy_targets(y), None, None, None, None, 1.0, 0.0, 0.0, 0.0, temperature)
        return loss

    def encoder_feature_distillation(self, student_features, teacher_features):
        """0.6*MSE(global mean) + 0.4*MSE(softmax-pooled) (reference :56-94); needs logits only for the batch size."""
        B = student_features.shape[0]
        y = torch.zeros(1, B, 8, device=student_features.device)
        loss, _ = self._run(y, y, self._dummy_targets(y), student_features, teacher_features, None, None, 0.0, 1.0, 0.0, 0.0, 1.0)
        return loss

    def decoder_hidden_state_distillation(self, student_hiddens, teacher_hiddens):
        """mean_t[0.7*MSE + 0.3*(1-cos)] (reference :96-136); 0 when either side is None."""
        if student_hiddens is None or teacher_hiddens is None:
            return 0.0
        hs, ht = _stack_hidden(student_hiddens), _stack_hidden(teacher_hiddens)
        y = torch.zeros(1, hs.shape[1], 8, device=hs.device)
        loss, _ = self._run(y, y, self._dummy_targets(y), None, None, hs, ht, 0.0, 0.0, 1.0, 0.0, 1.0)
        return loss


class FeatureProjector(nn.Module):
    """Teacher -> student feature space: Linear/ReLU/Dropout(0.1)/LayerNorm on the channel axis, then
    AdaptiveAvgPool1d on the token axis (reference :203-252)."""

    def __init__(self, teacher_dim, student_dim, teacher_seq_len=197, student_seq_len=64):
        super().__init__()
        self.teacher_dim = teacher_dim
        self.student_dim = student_dim
        self.teacher_seq_len = teacher_seq_len
        self.student_seq_len = student_seq_len
        if teacher_dim != student_dim:
            self.feature_projection = nn.Sequential(nn.Linear(teacher_dim, student_dim), nn.ReLU(), nn.Dropout(0.1),
                                                    nn.LayerNorm(student_dim))
        else:
            self.feature_projection = nn.Identity()
        self.seq_projection = nn.AdaptiveAvgPool1d(student_seq_len) if teacher_seq_len != student_seq_len else nn.Identity()

    def forward(self, features):
        """(B, teacher_seq_len, teacher_dim) -> (B, student_seq_len, student_dim) fp32, through b2c_projector_forward /
        _backward (parameters stay in the reference's stock submodules).  Gradients flow to the parameters; the teacher
        features are treated as data (the reference's TeacherWrapper produces them under no_grad)."""
        p = 0.1 if (self.training and self.teacher_dim != self.student_dim) else 0.0
        self._step = getattr(self, "_step", 0) + 1
        seed = (torch.initial_seed() + 0xA24BAED4963EE407 * self._step) & 0xFFFFFFFFFFFFFFFF if p > 0 else 0
        dt = torch.bfloat16 if torch.is_autocast_enabled() else getattr(self, "compute_dtype", torch.float32)
        named = dict(self.named_parameters())
        params = [named[k] for k in _ops.PROJ_PARAM_ORDER] if self.teacher_dim != self.student_dim else []
        return _ops.ProjectorFunction.apply(features, dt, p, seed, self.student_seq_len, self.student_dim,
                                            getattr(self, "b2c_options", None), *params)


class TeacherWrapper(nn.Module):
    """Frozen teacher in eval mode -> {'logits','encoder_features','hidden_states': None}, fp32 (reference :255-292)."""

    def __init__(self, teacher_model):
        super().__init__()
        self.teacher = teacher_model
        self.teacher.eval()
        for prm in self.teacher.parameters():
            prm.requires_grad = False

    def forward(self, images, captions):
        with torch.no_grad():
            images = images.float()
            captions = captions.long()
            logits = self.teacher(images, captions)
            feats = self.teacher.encoder_projection(self.teacher.encoder.forward_features(images))
            return {"logits": logits.float(), "encoder_features": feats.float(), "hidden_states": None}


def create_feature_projectors(teacher_model, student_model):
    """{'encoder': FeatureProjector(teacher enc dim -> student embed, 197 -> student tokens), 'hidden': ...} (reference :295-340)."""
    proj = teacher_model.encoder_projection
    if hasattr(proj, "out_features"):
        teacher_dim = proj.out_features
    elif hasattr(proj, "in_features"):
        teacher_dim = proj.in_features
    else:
        teacher_dim = teacher_model.encoder.num_features
    student_dim = student_model.embed_size
    if hasattr(student_model.encoder, "adaptive_pool"):
        size = student_model.encoder.adaptive_pool.output_size
        student_tokens = size[0] * size[1] if isinstance(size, tuple) else size * size
    else:
        student_tokens = 64
    print(f"Creating encoder projector: {teacher_dim} -> {student_dim}, seq_len: 197 -> {student_tokens}")
    projectors = {"encoder": FeatureProjector(teacher_dim, student_dim, teacher_seq_len=197, student_seq_len=student_tokens)}
    teacher_hidden = getattr(teacher_model, "embed_size", 512)
    print(f"Creating hidden projector: {teacher_hidden} -> {student_model.hidden_size}")
    projectors["hidden"] = FeatureProjector(teacher_hidden, student_model.hidden_size)
    return projectors


def validate_distillation_setup(teacher_model, student_model, sample_batch):
    """Dry run: teacher + student forward, projectors, one loss (reference :343-394). Returns (projectors, loss module)."""
    print("Validating distillation setup...")
    images, captions = sample_batch
    teacher_outputs = TeacherWrapper(teacher_model)(images.float(), captions.long())
    logits, enc, hiddens, _ = student_model(images, captions)
    student_outputs = {"logits": logits, "encoder_features": enc, "hidden_states": hiddens}
    print(f"Teacher logits shape: {teacher_outputs['logits'].shape}")
    print(f"Student logits shape: {student_outputs['logits'].shape}")
    print(f"Teacher encoder features shape: {teacher_outputs['encoder_features'].shape}")
    print(f"Student encoder features shape: {student_outputs['encoder_features'].shape}")
    projectors = create_feature_projectors(teacher_model, student_model)
    for key in projectors:
        projectors[key] = projectors[key].to(images.device)
    projected = projectors["encoder"](teacher_outputs["encoder_features"])
    print(f"Projected teacher features shape: {projected.shape}")
    distill_loss = DistillationLoss(vocab_size=teacher_outputs["logits"].size(-1))
    teacher_outputs["encoder_features"] = projected
    _, loss_dict = distill_loss(student_outputs, teacher_outputs, captions)
    print("Distillation loss validation successful!")
    print(f"Loss components: {loss_dict}")
    return projectors, distill_loss


def compute_bleu_score(predicted_tokens, target_tokens, vocab):
    """Set-overlap 'BLEU-1' used for monitoring (reference :398-409): |pred ∩ target| / |target| over non-special words."""
    special = (0, 1, 2)
    pred = {vocab.itos[i] for i in predicted_tokens if i not in special}
    target = {vocab.itos[i] for i in target_tokens if i not in special}
    if not any(i not in special for i in target_tokens):
        return 0.0
    return len(pred & target) / len(target)


def log_training_progress(epoch, batch_idx, loss_dict, learning_rate, total_batches):
    """Print the loss components every 50 batches (reference :412-422)."""
    if batch_idx % 50 != 0:
        return
    print(f"Epoch {epoch}, Batch {batch_idx}/{total_batches}")
    print(f"  LR: {learning_rate:.6f}")
    for label, key in (("Total Loss", "total_loss"), ("CE Loss", "ce_loss"), ("Token KD", "token_kd_loss"),
                       ("Feature KD", "feature_kd_loss"), ("Hidden KD", "hidden_kd_loss")):
        print(f"  {label}: {loss_dict[key]:.4f}")
    print("-" * 50)
