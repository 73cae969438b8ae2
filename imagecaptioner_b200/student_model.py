"""Drop-in for the reference's ``src/student_model.py`` on the KD hot path.

Same classes, constructor arguments, attribute / submodule names and ``state_dict`` keys as the
reference (``/root/reference/src/student_model.py``), so ``train_student_kd.py`` and
``evaluate_student.py`` run unchanged and reference checkpoints load with ``load_state_dict``.
What differs is the body of the hot path: ``LSTMDecoder.forward`` (reference :205-256) and the
greedy loop of ``CaptioningStudent.caption_image`` (reference :314-381) are single calls into the
hand-written sm_100a kernels behind ``include/b2c.h``.  The (once per sequence) ``AttentionRefinement``
block keeps its parameters in the reference's stock submodules (same ``state_dict`` keys) but computes
through ``b2c_refinement_forward`` / ``_backward`` (SURVEY.md §8f row 1); only the ResNet encoder stays a
stock ``torch.nn`` module — SURVEY.md §8 keeps it out of the path.  ``LSTMDecoder.forward`` also takes the
reference's optional ``hidden=(h0, c0)`` initial state (``b2c_decoder_set_initial_state``).

Precision mode of the decoder: bf16 (tcgen05 tensor-core tiles) when called under
``torch.autocast`` — the reference trains under fp16 autocast, ``train_student_kd.py:271`` — or when
``decoder.compute_dtype = torch.bfloat16``; fp32 (parity mode) otherwise.
"""
from __future__ import annotations

import os

from typing import List

import torch
import torch.nn as nn

from . import _ops


class CNNEncoder(nn.Module):
    """ResNet-50 trunk -> 7x7 pool -> Linear/ReLU/Dropout/LayerNorm -> (B,49,E)  (reference :8-69).

    Outside the hot path (BASELINE.json north_star): kept so checkpoints and the optimizer groups of
    train_student_kd.py:219-228 line up.  Without network access the ImageNet weights cannot be
    downloaded; the trunk is then randomly initialised and a warning is printed."""

    def __init__(self, embed_size=256, fine_tune=True):
        super().__init__()
        import torchvision.models as models
        try:
            trunk = models.resnet50(weights=models.ResNet50_Weights.IMAGENET1K_V1)
        except Exception as exc:  # offline box
            print(f"[b2c] ImageNet weights unavailable ({type(exc).__name__}); ResNet-50 trunk randomly initialised")
            trunk = models.resnet50(weights=None)
        self.resnet = nn.Sequential(*list(trunk.children())[:-2])
        if fine_tune:
            for idx, child in enumerate(self.resnet.children()):
                for prm in child.parameters():
                    prm.requires_grad = idx >= 6          # conv1..layer2 frozen, layer3/4 trainable
        self.adaptive_pool = nn.AdaptiveAvgPool2d((7, 7))
        self.projection = nn.Sequential(nn.Linear(2048, embed_size), nn.ReLU(), nn.Dropout(0.2), nn.LayerNorm(embed_size))
        self.embed_size = embed_size

    def forward(self, images):
        fmap = self.adaptive_pool(self.resnet(images))                  # (B,2048,7,7)
        tokens = fmap.flatten(2).transpose(1, 2)                        # (B,49,2048)
        return self.projection(tokens)


class PrecomputedFeatures(nn.Module):
    """Stand-in encoder for runs that feed (B,49,E) features directly (benchmarks, parity tests): the
    north_star keeps the ResNet/ViT encoders outside the path.  Exposes ``adaptive_pool`` because
    create_feature_projectors reads ``encoder.adaptive_pool.output_size`` (reference distillation_utils.py:313-319)."""

    def __init__(self, embed_size=256, grid=7):
        super().__init__()
        self.adaptive_pool = nn.AdaptiveAvgPool2d((grid, grid))
        self.embed_size = embed_size

    def forward(self, features):
        if features.dim() == 2:
            features = features.unsqueeze(0)
        return features


class AttentionRefinement(nn.Module):
    """One post-norm self-attention block over the 49 tokens (reference :72-118)."""

    def __init__(self, embed_size, num_heads=4):
        super().__init__()
        self.embed_size = embed_size
        self.num_heads = num_heads
        self.attention = nn.MultiheadAttention(embed_dim=embed_size, num_heads=num_heads, dropout=0.1, batch_first=True)
        self.ffn = nn.Sequential(nn.Linear(embed_size, embed_size * 2), nn.ReLU(), nn.Dropout(0.1), nn.Linear(embed_size * 2, embed_size))
        self.norm1 = nn.LayerNorm(embed_size)
        self.norm2 = nn.LayerNorm(embed_size)

    def forward(self, features):
        """(B,S,E) -> (B,S,E).  The parameters live in the reference's stock submodules (state_dict compatible); the
        computation is one C-ABI call each way (b2c_refinement_forward / _backward).  bf16 under autocast, fp32 otherwise."""
        p = 0.1 if self.training else 0.0            # the reference's attention / FFN dropout
        self._step = getattr(self, "_step", 0) + 1
        seed = (torch.initial_seed() + 0xD1B54A32D192ED03 * self._step) & 0xFFFFFFFFFFFFFFFF if p > 0 else 0
        dt = torch.bfloat16 if torch.is_autocast_enabled() else getattr(self, "compute_dtype", torch.float32)
        named = dict(self.named_parameters())
        return _ops.RefinementFunction.apply(features, dt, p, seed, self.num_heads, getattr(self, "b2c_options", None),
                                             *[named[k] for k in _ops.REFINE_PARAM_ORDER])


class HiddenStateList(list):
    """The reference returns a Python list of T (B,H) tensors; this list also remembers the single
    (T,B,H) buffer they are views of so the loss kernel can take it without a stack copy."""
    stacked = None


class LSTMDecoder(nn.Module):
    """Attention-LSTM caption decoder (reference :121-256).  Parameters live in the same stock modules
    as the reference (same names, shapes, initialisers, gate order); the computation does not."""

    def __init__(self, vocab_size, embed_size=256, hidden_size=512, num_layers=2, dropout=0.2):
        super().__init__()
        if not 1 <= num_layers <= _ops.B2C_MAX_LAYERS:
            raise ValueError(f"num_layers={num_layers} outside [1,{_ops.B2C_MAX_LAYERS}]")
        self.embed_size = embed_size
        self.hidden_size = hidden_size
        self.num_layers = num_layers
        self.vocab_size = vocab_size
        self.dropout_p = float(dropout)
        self.compute_dtype = torch.float32          # bf16 under autocast or when set explicitly
        self.embedding = nn.Embedding(vocab_size, embed_size)
        nn.init.uniform_(self.embedding.weight, -0.1, 0.1)
        self.attention = nn.Linear(hidden_size + embed_size, embed_size)
        self.attention_combine = nn.Linear(embed_size * 2, embed_size)
        self.lstm = nn.LSTM(input_size=embed_size, hidden_size=hidden_size, num_layers=num_layers,
                            dropout=dropout if num_layers > 1 else 0, batch_first=True)
        self.output_projection = nn.Sequential(nn.Linear(hidden_size, embed_size), nn.ReLU(), nn.Dropout(dropout),
                                               nn.Linear(embed_size, vocab_size))
        for name, prm in self.lstm.named_parameters():
            if "weight_ih" in name:
                nn.init.xavier_uniform_(prm.data)
            elif "weight_hh" in name:
                nn.init.orthogonal_(prm.data)
            elif "bias" in name:
                prm.data.zero_()
        self._step = 0

    # ---- helpers
    def _param_list(self) -> List[torch.Tensor]:
        named = dict(self.named_parameters())
        return [named[k] for k in _ops.param_order(self.num_layers)]

    def _mode(self) -> torch.dtype:
        if torch.is_autocast_enabled():
            return torch.bfloat16
        return self.compute_dtype

    def init_hidden(self, batch_size, device):
        shape = (self.num_layers, batch_size, self.hidden_size)
        return torch.zeros(shape, device=device), torch.zeros(shape, device=device)

    @torch.no_grad()
    def attention_mechanism(self, hidden, image_features):
        """context (B,E), attention weights (B,S) of one step (reference :173-203), stand-alone accessor
        (inference only; inside forward / greedy the same kernel runs as part of the fused step)."""
        return _ops.attention_step(hidden, image_features, self.attention.weight, self.attention.bias, self._mode())

    def prepare(self, captions, num_tokens):
        """Start the part of `forward` that does not need the image features (operand packing, embedding rows, the embedding
        half of layer 0's gates) on a side stream; pass the handle to forward(..., prepared=handle)."""
        return _ops.decoder_prepare(captions, num_tokens, self._mode(), self.num_layers, self._param_list())

    def forward(self, image_features, captions, hidden=None, prepared=None):
        """image_features (B,S,E), captions (T,B) -> outputs (T,B,V), hidden_states [T x (B,H)], attention [T x (B,S)]."""
        if hidden is not None:
            # reference :205 / :219-222: (h0, c0), each (num_layers, B, hidden_size), seed the recurrence instead of init_hidden's zeros.
            # The state is an input here, not a differentiable one (nothing in the reference passes it, let alone trains through it).
            if any(getattr(t, "requires_grad", False) for t in hidden):
                raise NotImplementedError("gradients with respect to the initial `hidden` state are not produced; pass detached tensors")
            hidden = (hidden[0], hidden[1])
        p = self.dropout_p if self.training else 0.0
        self._step += 1
        seed = (torch.initial_seed() + 0x9E3779B97F4A7C15 * self._step) & 0xFFFFFFFFFFFFFFFF if p > 0 else 0
        logits, hid, attw = _ops.DecoderFunction.apply(image_features, captions, self._mode(), p, seed, self.num_layers, prepared,
                                                       getattr(self, "b2c_options", None), hidden, *self._param_list())
        hidden_states = HiddenStateList(hid.unbind(0))
        hidden_states.stacked = hid
        return logits, hidden_states, list(attw.unbind(0))

    @torch.no_grad()
    def greedy(self, image_features, max_length, start_id=1, end_id=2, use_graph=None):
        """Batched greedy decode of already-refined features -> tokens (max_length,B) int64, lengths (B) int32.

        One decode is ~9 small kernels per token with the argmax fed back on the device; issued eagerly it is bound by host
        launch latency, so for batches >= 64 (or use_graph=True) the whole decode is captured once per (shape, dtype, ids) into
        a CUDA graph over a static feature buffer and replayed.  The parameters are read through their pointers at replay
        time, so in-place weight updates are seen; the returned tensors are copies of the graph's static outputs."""
        B = image_features.shape[0]
        if use_graph is None:
            use_graph = B >= 64
        if not use_graph:
            return _ops.greedy_decode(image_features, self._param_list(), self.num_layers, max_length, start_id, end_id, self._mode())
        plist = self._param_list()
        key = (tuple(image_features.shape), int(max_length), int(start_id), int(end_id), self._mode(), image_features.device,
               tuple(p.data_ptr() for p in plist))
        cache = self.__dict__.setdefault("_greedy_graphs", {})
        ent = cache.get(key)
        if ent is None:
            static_feats = image_features.detach().float().clone()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                      # warm-up outside capture (lazy module/attribute initialisation)
                _ops.greedy_decode(static_feats, plist, self.num_layers, max_length, start_id, end_id, self._mode())
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                toks, lens = _ops.greedy_decode(static_feats, plist, self.num_layers, max_length, start_id, end_id, self._mode())
            if len(cache) >= 8:
                cache.clear()
            ent = cache[key] = (graph, static_feats, toks, lens)
        graph, static_feats, toks, lens = ent
        static_feats.copy_(image_features)
        graph.replay()
        return toks.clone(), lens.clone()


class CaptioningStudent(nn.Module):
    """Encoder -> optional refinement -> decoder (reference :259-381)."""

    def __init__(self, vocab_size, embed_size=256, hidden_size=512, num_layers=2, dropout=0.2, use_attention_refinement=True,
                 encoder=None):
        super().__init__()
        self.vocab_size = vocab_size
        self.embed_size = embed_size
        self.hidden_size = hidden_size
        # `encoder` is an extension (default = the reference's ResNet-50 encoder): pass PrecomputedFeatures() to feed features
        self.encoder = CNNEncoder(embed_size=embed_size, fine_tune=True) if encoder is None else encoder
        self.use_attention_refinement = use_attention_refinement
        self.overlap_decoder_prepare = os.environ.get("B2C_OVERLAP_PREPARE", "1") != "0"
        if use_attention_refinement:
            self.attention_refinement = AttentionRefinement(embed_size=embed_size)
        self.decoder = LSTMDecoder(vocab_size=vocab_size, embed_size=embed_size, hidden_size=hidden_size,
                                   num_layers=num_layers, dropout=dropout)

    def forward(self, images, captions):
        """-> (outputs (T,B,V), encoder_features (B,49,E) UN-refined, hidden_states list, attention_weights list)."""
        encoder_features = self.encoder(images)
        prepared = None
        if self.use_attention_refinement and encoder_features.is_cuda and self.overlap_decoder_prepare:
            # the decoder's feature-independent preamble runs on a side stream underneath the refinement block
            prepared = self.decoder.prepare(captions, encoder_features.shape[1])
        refined = self.attention_refinement(encoder_features) if self.use_attention_refinement else encoder_features
        outputs, hidden_states, attention_weights = self.decoder(refined, captions, prepared=prepared)
        return outputs, encoder_features, hidden_states, attention_weights

    def supports_fused_validation(self) -> bool:
        """The logits-free validation forward exists in bf16 mode (autocast, or decoder.compute_dtype = bfloat16), for any vocabulary
        size (the epilogue reads teacher rows that do not start on a 16-byte boundary with plain loads)."""
        return self.decoder._mode() == torch.bfloat16

    @torch.no_grad()
    def forward_validation(self, images, captions, teacher_logits, targets, temperature):
        """validate_student_model's student forward (reference src/train_student_kd.py:56) fused with the token part of the loss:
        -> (rows (2, T*B) per-row [KL, CE] partials, predicted tokens (T,B) = logits.argmax(-1), encoder_features (B,49,E) un-refined,
        hidden_states list, attention_weights list).  No (T,B,V) logits tensor exists at any point (b2c_decoder_forward_eval)."""
        encoder_features = self.encoder(images)
        refined = self.attention_refinement(encoder_features) if self.use_attention_refinement else encoder_features
        hid, attw, rows, pred = _ops.decoder_forward_eval(refined, captions, teacher_logits, targets, temperature,
                                                          self.decoder.num_layers, self.decoder._param_list())
        hidden_states = HiddenStateList(hid.unbind(0))
        hidden_states.stacked = hid
        return rows, pred, encoder_features, hidden_states, list(attw.unbind(0))

    @torch.no_grad()
    def caption_images(self, images, vocabulary, max_length=20):
        """Batched form of caption_image: one device-side greedy decode for the whole batch."""
        self.eval()
        device = next(self.parameters()).device
        feats = self.encoder(images.to(device))
        if self.use_attention_refinement:
            feats = self.attention_refinement(feats)
        start = vocabulary.stoi.get("<START>", vocabulary.stoi["<UNK>"])
        end = vocabulary.stoi.get("<END>", -1)
        tokens, lengths = self.decoder.greedy(feats, max_length, start, end)
        tokens, lengths = tokens.cpu(), lengths.cpu()              # ONE device->host copy for the batch
        return [[vocabulary.itos[int(tokens[t, b])] for t in range(int(lengths[b]))] for b in range(tokens.shape[1])]

    def caption_image(self, image, vocabulary, max_length=20, temperature=1.0):
        """Greedy caption of one image as a list of words (temperature rescales logits and cannot change the argmax)."""
        if image.dim() == 3:
            image = image.unsqueeze(0)
        return self.caption_images(image, vocabulary, max_length=max_length)[0]


def count_parameters(model):
    total = sum(p.numel() for p in model.parameters())
    trainable = sum(p.numel() for p in model.parameters() if p.requires_grad)
    return total, trainable
