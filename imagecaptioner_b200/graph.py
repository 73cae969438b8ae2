"""Whole-step CUDA graph for the KD training step.

One KD step launches several hundred small kernels (T serial decode steps, forward and backward); issued
eagerly the step is bound by host launch latency, not by the GPU.  ``GraphedKDStep`` captures the complete step —
student forward (refinement + decoder), FeatureProjector, DistillationLoss, backward, gradient all-reduce,
global-norm clip and AdamW — into ONE ``torch.cuda.CUDAGraph`` over static input buffers and replays it with a
single launch per step (SURVEY.md §7.3 item 1: "CUDA Graph over the whole sequence at minimum").

``optimizer`` is either ``optim.FlatAdamW`` (native: the reference's two clip groups and three LR groups on flat buffers,
``max_grad_norm`` then comes from the optimizer) or any capturable ``torch.optim`` optimizer (then one global-norm clip over
the whole flat buffer precedes ``optimizer.step()``).

The step structure is the reference's training loop body (src/train_student_kd.py:262-303) with the encoders
outside the path: the caller provides encoder features, captions, targets and the teacher's outputs.

Variable-length batches (``max_steps=T_cap``): the reference's loader pads every batch to its own longest caption, so T changes
from batch to batch.  The graph is then captured once with (T_cap, B, ...) buffers and a device step count; ``load()`` takes any
batch with 1 <= T <= T_cap and the replay computes exactly the loss, gradients and update of that T-step batch (padding the batch
to T_cap instead would not: token KD is a mean over all T*B rows and hidden KD a mean over steps).

Half-precision teacher outputs: the static buffers take the example batch's dtypes.  With bf16 / fp16 teacher_logits,
teacher_features and teacher_hiddens in the example, the captured kernels read them in that precision and widen them exactly to
fp32 in registers (the same loss parts and gradients as for their fp32 upcasts), the graph holds no conversion of them, and load()
copies half the teacher bytes.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import torch

from . import _ops
from .ddp import FlatGradAllReducer


class GraphedKDStep:
    INPUT_KEYS = ("encoder_features", "captions_input", "targets", "teacher_logits", "teacher_features", "teacher_hiddens")
    TIME_KEYS = ("captions_input", "targets", "teacher_logits", "teacher_hiddens")      # (T, B, ...): the time axis first

    def __init__(self, model, projector, loss_module, optimizer, reducer: Optional[FlatGradAllReducer], example: Dict[str, torch.Tensor],
                 max_grad_norm: float = 1.0, autocast_dtype: Optional[torch.dtype] = torch.bfloat16, use_graph: bool = True,
                 warmup_steps: int = 3, direct_grads: bool = True, max_steps: Optional[int] = None):
        self.model, self.projector, self.loss_module = model, projector, loss_module
        self._native_opt = hasattr(optimizer, "flat_param") and hasattr(optimizer, "reducer")     # optim.FlatAdamW
        if self._native_opt:
            if reducer is None:
                reducer = optimizer.reducer
            if reducer is not optimizer.reducer:
                raise ValueError("a FlatAdamW optimizer brings its own gradient buffer: pass reducer=None or optimizer.reducer")
        self.optimizer, self.reducer = optimizer, reducer
        # native optimizer: the 1/world of the gradient average is applied inside the update kernel instead of a pass of its own
        self._fold_avg = self._native_opt and reducer.world_size > 1
        if self._fold_avg:
            optimizer.fold_average(reducer.world_size)
        self.max_grad_norm = max_grad_norm
        self.autocast_dtype = autocast_dtype
        # max_steps: static (max_steps, B, ...) buffers and a device step count (steps[0] = T of the loaded batch) that the decoder
        # and the loss read at replay time (CallOptions.steps_dev); None: buffers of the example's shape, every batch that shape
        self.max_steps = max_steps
        self.steps = None
        if max_steps is None:
            self.static = {k: example[k].clone() for k in self.INPUT_KEYS if example.get(k) is not None}
        else:
            T = example["captions_input"].shape[0]
            if not 1 <= T <= max_steps:
                raise ValueError(f"the example batch has T={T} steps, max_steps={max_steps}")
            self.static = {}
            for k in self.INPUT_KEYS:
                src = example.get(k)
                if src is None:
                    continue
                if k in self.TIME_KEYS:
                    self.static[k] = torch.zeros((max_steps,) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
                else:
                    self.static[k] = src.clone()
            self.steps = torch.zeros(1, dtype=torch.int32, device=example["targets"].device)
            self.load(example, non_blocking=False)
        self.static["encoder_features"].requires_grad_(True)
        self.out5 = None
        self.graph = None          # forward + loss + backward (+ clip + AdamW when there is a single rank)
        self.graph_opt = None      # clip + AdamW, a second graph when a gradient all-reduce sits in between
        self.world = reducer.world_size
        self._side = torch.cuda.Stream()
        self._aux = torch.cuda.Stream()
        self._aux_used = False
        self._overlap = False
        self._capturing = False
        self.high_priority_chain = os.environ.get("B2C_CHAIN_PRIORITY", "1") != "0"
        self.defer_weight_grad_join = os.environ.get("B2C_DEFER_JOIN", "1") != "0"
        self.background_ctas = int(os.environ.get("B2C_BG_CTAS", "10"))       # CTA budget of GEMMs that overlap a recurrence (0 = no limit)
        # every trainable parameter here gets exactly one gradient per step from one native backward call, so the kernels may
        # write it directly into the flat all-reduce buffer (saves ~35 accumulate kernels + the buffer zeroing per step)
        self.direct_grads = direct_grads
        loss_module.assume_unit_grad = True      # _fwd_bwd calls loss.backward() with the implicit grad_output of exactly 1
        # Per-model call options (nothing process-global): gradient destinations, deferred weight-gradient join, the event hook
        # behind the decoder backward, and the device-side dropout step counter.  They are attached to the modules only for the
        # duration of this object's own forward/backward (see _fwd_bwd), so an eager loop on the same model is unaffected.
        dev = self.static["targets"].device
        self.step_counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self._opts = _ops.CallOptions(grad_dest=reducer.grad_views() if direct_grads else None, seed_dev=self.step_counter, steps_dev=self.steps)
        # Data parallel: NCCL stays OUTSIDE the graphs (graph 1 = forward + loss + backward, graph 2 = clip + AdamW); the two
        # exchanges (non-PAD count, flat gradient buffer) are issued eagerly around / alongside graph 1, see overlap_comm below.
        # B2C_FAKE_DP=1: exercise the multi-rank control flow (two graphs, overlapped exchanges) on ONE GPU with an identity in
        # place of each collective -- used by the tests, which cannot run NCCL.
        self._fake_dp = self.world == 1 and os.environ.get("B2C_FAKE_DP", "0") == "1"
        self._multi = self.world > 1 or self._fake_dp
        self.nval = torch.zeros(1, dtype=torch.int32, device=self.static["targets"].device) if self._multi else None
        # single rank under capture: the non-PAD count is taken off the main chain (it only depends on the targets): counted on the
        # projector's side stream at the start of the step instead of between the vocabulary head and the token loss
        self._nval_single = torch.zeros(1, dtype=torch.int32, device=self.static["targets"].device) if not self._multi else None
        # Overlapped exchanges (graph mode, multi-rank): the collectives run on a communication stream, tied to the graph by
        # EXTERNAL events -- the non-PAD count is all-reduced under the forward (graph 1 waits for it just before the loss) and
        # the decoder's gradient segment (90 % of the bytes) is all-reduced under the refinement backward (graph 1 records an
        # event right after b2c_decoder_backward).
        self.overlap_comm = use_graph and self._multi and os.environ.get("B2C_OVERLAP_COMM", "1") != "0"
        self._early = self._early_segment() if self.overlap_comm else None
        if self.overlap_comm:
            self._comm = torch.cuda.Stream()
            self._ev_count = torch.cuda.Event(external=True)
            self._ev_dec = torch.cuda.Event(external=True)
        if use_graph:
            self._capture(warmup_steps)

    # ---- collectives (identity in the single-GPU fake mode)
    def _all_reduce(self, t):
        if self.world > 1:
            torch.distributed.all_reduce(t, group=self.loss_module.process_group)
        else:
            t.add_(0)

    def _early_segment(self):
        """[a, b) of the flat gradient buffer that holds exactly the decoder's parameters, or None if they are not contiguous."""
        dec = {id(p) for p in self.model.decoder.parameters() if p.requires_grad}
        spans = [(o, o + p.numel()) for p, o in zip(self.reducer.params, self.reducer.offsets) if id(p) in dec]
        if not spans or len(spans) != len(dec):
            return None
        a, b = min(s[0] for s in spans), max(s[1] for s in spans)
        inside = [p for p, o in zip(self.reducer.params, self.reducer.offsets) if a <= o < b and id(p) not in dec]
        return None if inside else (a, b)

    # ---- the step body (eager or under capture)
    def _pre(self):
        if self._multi:
            _ops.count_valid(self.static["targets"], self.loss_module.vocab_size or 2 ** 31 - 1, out=self.nval)
            self._all_reduce(self.nval)
            self.loss_module.n_valid_global = self.nval

    def _modules(self):
        mods = [self.model.decoder, self.projector]
        if getattr(self.model, "use_attention_refinement", False):
            mods.append(self.model.attention_refinement)
        return mods

    def _attach_options(self):
        o = self._opts
        # Single rank: the weight-gradient branch of b2c_decoder_backward (side stream) is joined AFTER the whole backward, so the
        # refinement backward overlaps it instead of waiting 0.26 ms for it (the parameters' gradients are first read by the
        # optimizer).  Multi-rank with the overlapped exchange: the communication stream needs the decoder's gradients right behind
        # the call, so the hook below joins the side branch on the MAIN stream only when it has to record the event there.
        early = self._capturing and self.overlap_comm and self._early is not None
        o.defer_join = self.defer_weight_grad_join and self.direct_grads and (not self._multi or early)
        o.after_backward = self._after_decoder_backward if early else None
        # under capture the projector (forward and backward) lives on a side stream next to the decoder's recurrences
        o.background_ctas = self.background_ctas if self._overlap else 0
        for m in self._modules():
            m.b2c_options = o
        if self.steps is not None:
            self.loss_module.b2c_options = o        # the KD loss reads steps_dev (rows / steps past it: no loss, zero gradient)

    def _after_decoder_backward(self):
        """Runs right behind b2c_decoder_backward (autograd thread, capture stream).  The communication stream may start the
        all-reduce of the decoder's gradient segment once BOTH the main chain up to here and the library's weight-gradient side
        branch are done; the main chain itself does not wait for that branch (the refinement backward follows immediately), so the
        event is recorded on an auxiliary captured stream that joins the two."""
        main = torch.cuda.current_stream()
        if self._opts.join_pending:
            self._opts.join_pending = False
            self._aux.wait_stream(main)
            with torch.cuda.stream(self._aux):
                _ops.join_side_work()
                self._ev_dec.record()
            self._aux_used = True
        else:
            self._ev_dec.record()

    def _detach_options(self):
        for m in self._modules():
            m.b2c_options = None
        if self.steps is not None:
            self.loss_module.b2c_options = None

    def release(self):
        """Drop the graphs and every hook this object attached (the model can then be trained eagerly, e.g. with gradient
        accumulation, without its gradients being redirected into the flat buffer)."""
        self._detach_options()
        self.graph = self.graph_opt = None

    def _dropout_active(self):
        return any(m.training for m in self._modules())

    def _fwd_bwd(self):
        inp = self.static
        feats = inp["encoder_features"]
        if feats.grad is not None:
            feats.grad = None
        self._attach_options()
        if self._dropout_active():
            _ops.bump_counter(self.step_counter)     # a fresh dropout mask per step, also when the step is a graph replay
        ctx = torch.autocast("cuda", dtype=self.autocast_dtype) if self.autocast_dtype is not None else torch.autocast("cuda", enabled=False)
        # The projector does not depend on the student: it runs on a side stream underneath the decoder's latency-bound
        # recurrence (fork / join are recorded as parallel branches by the graph capture).
        # (only under capture, where every buffer lives in the graph's private pool; eagerly the projector stays in stream order)
        if self._overlap:
            main = torch.cuda.current_stream()
            self._side.wait_stream(main)
            if self._nval_single is not None:
                with torch.cuda.stream(self._side):
                    _ops.count_valid(inp["targets"], self.loss_module.vocab_size or 2 ** 31 - 1, out=self._nval_single)
                self.loss_module.n_valid_global = self._nval_single
            with torch.cuda.stream(self._side), ctx:
                tproj = self.projector(inp["teacher_features"])
            with ctx:                                                  # the reference's loop runs under autocast (train_student_kd.py:271)
                outputs, enc, hids, _ = self.model(feats, inp["captions_input"])
            main.wait_stream(self._side)
        else:
            with ctx:
                outputs, enc, hids, _ = self.model(feats, inp["captions_input"])
                tproj = self.projector(inp["teacher_features"])
        if self._capturing and self.overlap_comm:
            torch.cuda.current_stream().wait_event(self._ev_count)      # external event: the count all-reduce of THIS step
        loss, out5 = self.loss_module.forward_device(
            {"logits": outputs, "encoder_features": enc, "hidden_states": hids},
            {"logits": inp["teacher_logits"], "encoder_features": tproj, "hidden_states": inp.get("teacher_hiddens")},
            inp["targets"])
        if self.direct_grads:
            self.reducer.detach_grads()          # backward kernels write every parameter gradient straight into the flat buffer
        else:
            self.reducer.zero_grad()
        try:
            loss.backward()
        finally:
            self._detach_options()
            if self._nval_single is not None:
                self.loss_module.n_valid_global = None      # the captured kernels hold the pointer; an eager use of the loss module counts itself
            if self._opts.join_pending:          # the decoder backward deferred its weight-gradient join (B2C_BWD_DEFER_JOIN)
                self._opts.join_pending = False
                _ops.join_side_work()
            if self._aux_used:                   # the auxiliary branch that carries the event record rejoins the capture stream
                self._aux_used = False
                torch.cuda.current_stream().wait_stream(self._aux)
        if self.direct_grads:
            self.reducer.attach_views()          # the flat buffer is authoritative (the kernels wrote into it), whatever autograd kept
        return out5

    def _clip_and_update(self):
        if self._native_opt:                                           # optim.FlatAdamW: unscale + per-group clip + AdamW, 2 launches
            self.optimizer.step()
            return
        if self.max_grad_norm is not None:                             # clip_grad_norm_ on the flat buffer, no host sync
            gn = self.reducer.flat.norm()
            self.reducer.flat.mul_(torch.clamp(self.max_grad_norm / (gn + 1e-6), max=1.0))
        self.optimizer.step()

    def _exchange_grads(self):
        if self.world > 1:
            if self._fold_avg:
                self._all_reduce(self.reducer.flat)
            else:
                self.reducer.allreduce()
        elif self._fake_dp:
            self._all_reduce(self.reducer.flat)

    def _body(self):
        self._pre()
        out5 = self._fwd_bwd()
        self._exchange_grads()
        self._clip_and_update()
        return out5

    def _capture(self, warmup_steps):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup_steps):
                self.out5 = self._body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._pre()
        torch.cuda.synchronize()
        if self.overlap_comm:
            self._ev_count.record()                                      # the wait node needs a recorded event at capture time
        self.graph = torch.cuda.CUDAGraph()
        self._overlap = True
        self._capturing = True
        # Captured on a HIGH-priority stream: kernel nodes keep the priority of the stream they were captured from, so the
        # latency-bound main chain (the recurrence) is scheduled ahead of the throughput work forked onto the default-priority
        # side streams (projector, weight gradients), which then only fills the SMs the chain leaves idle.
        cap = torch.cuda.Stream(priority=-1) if self.high_priority_chain else torch.cuda.Stream()
        if not self._multi:
            with torch.cuda.graph(self.graph, stream=cap):
                self.out5 = self._fwd_bwd()
                self._clip_and_update()
        else:
            with torch.cuda.graph(self.graph, stream=cap):
                self.out5 = self._fwd_bwd()
            self._exchange_grads()
            self.graph_opt = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_opt, pool=self.graph.pool()):
                self._clip_and_update()
        self._overlap = False
        self._capturing = False

    def load(self, batch: Dict[str, torch.Tensor], non_blocking: bool = True) -> int:
        """Copy one step's inputs (host or device tensors) into the static buffers; returns the bytes copied.

        With max_steps: a batch of any T <= max_steps steps (captions_input, targets, teacher_logits and teacher_hiddens all of T
        steps).  It fills steps [0, T) of the time-indexed buffers, writes PAD (0) into the caption and target steps past T (they
        then add nothing to the non-PAD count), leaves the teacher's steps past T as they are (never read) and sets the device step
        count to T, all on the current stream."""
        if self.max_steps is None:
            n = 0
            with torch.no_grad():
                for k, dst in self.static.items():
                    src = batch[k]
                    dst.copy_(src, non_blocking=non_blocking)
                    n += src.numel() * src.element_size()
            return n
        T = int(batch["captions_input"].shape[0])
        if not 1 <= T <= self.max_steps:
            raise ValueError(f"batch of T={T} steps: this GraphedKDStep takes 1 <= T <= max_steps={self.max_steps}")
        for k in self.TIME_KEYS:
            if k in self.static and batch[k].shape[0] != T:
                raise ValueError(f"{k} has {batch[k].shape[0]} steps, captions_input {T}")
        n = 0
        with torch.no_grad():
            for k, dst in self.static.items():
                src = batch[k]
                if k in self.TIME_KEYS:
                    dst[:T].copy_(src, non_blocking=non_blocking)
                    if k in ("captions_input", "targets") and T < self.max_steps:
                        dst[T:].zero_()
                else:
                    dst.copy_(src, non_blocking=non_blocking)
                n += src.numel() * src.element_size()
            self.steps.fill_(T)
        return n

    def step(self) -> torch.Tensor:
        """Run one KD step on the current contents of the static buffers -> device tensor
        [total, ce, token_kd, feature_kd, hidden_kd] (no host sync)."""
        if self.graph is None:
            self.out5 = self._body()
        elif not self._multi:
            self.graph.replay()
        elif not self.overlap_comm:
            self._pre()
            self.graph.replay()
            self._exchange_grads()
            self.graph_opt.replay()
        else:
            main, comm = torch.cuda.current_stream(), self._comm
            comm.wait_stream(main)                   # the previous step has consumed nval and the gradient buffer
            with torch.cuda.stream(comm):
                self._pre()                          # count + all-reduce under the forward
                self._ev_count.record()
            self.graph.replay()                      # waits for _ev_count before the loss; records _ev_dec after the decoder backward
            flat = self.reducer.flat
            if self._early is not None:
                a, b = self._early
                with torch.cuda.stream(comm):
                    comm.wait_event(self._ev_dec)
                    self._all_reduce(flat[a:b])      # decoder gradients, under the refinement backward
                if a > 0:
                    self._all_reduce(flat[:a])
                if b < flat.numel():
                    self._all_reduce(flat[b:])
                main.wait_stream(comm)
            else:
                self._all_reduce(flat)
            if self.world > 1 and not self._fold_avg:
                self.reducer.finish()
            self.graph_opt.replay()
        return self.out5
