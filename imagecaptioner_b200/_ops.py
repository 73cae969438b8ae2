"""ctypes binding of the b2c C ABI (include/b2c.h) + the autograd Functions built on it.

PyTorch is plumbing here (device memory, streams, autograd bookkeeping); every arithmetic
operation of the hot path runs in the hand-written sm_100a kernels of ``lib/libb2c.so``.
There is no CPU or eager fallback: a missing library or a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2C_LIB") or os.path.join(_HERE, "lib", "libb2c.so")      # B2C_LIB: A/B builds (development only)

B2C_MAX_LAYERS = 4
B2C_F32, B2C_BF16, B2C_F16 = 0, 1, 2          # B2C_F16: teacher operands only
B2C_WS_TRAIN, B2C_WS_DECODE, B2C_WS_ATTN, B2C_WS_REFINE, B2C_WS_PROJ = 0, 1, 2, 3, 4
ABI_VERSION = 5
B2C_BWD_DEFER_JOIN = 1

c_f32p = ctypes.c_void_p


class B2CShape(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("B", "T", "S", "E", "H", "L", "V")]


_PARAM_FIELDS = (
    [("embedding", c_f32p), ("attn_w", c_f32p), ("attn_b", c_f32p), ("comb_w", c_f32p), ("comb_b", c_f32p)]
    + [(n, c_f32p * B2C_MAX_LAYERS) for n in ("w_ih", "w_hh", "b_ih", "b_hh")]
    + [("out0_w", c_f32p), ("out0_b", c_f32p), ("out3_w", c_f32p), ("out3_b", c_f32p)]
)


class B2CParams(ctypes.Structure):
    _fields_ = _PARAM_FIELDS


class B2CGrads(ctypes.Structure):
    _fields_ = _PARAM_FIELDS


_REFINE_FIELDS = [(n, c_f32p) for n in ("in_w", "in_b", "out_w", "out_b", "ffn0_w", "ffn0_b", "ffn3_w", "ffn3_b", "n1_w", "n1_b", "n2_w", "n2_b")]
_PROJ_FIELDS = [(n, c_f32p) for n in ("w", "b", "ln_w", "ln_b")]


class B2CRefineParams(ctypes.Structure):
    _fields_ = _REFINE_FIELDS


class B2CRefineGrads(ctypes.Structure):
    _fields_ = _REFINE_FIELDS


class B2CProjParams(ctypes.Structure):
    _fields_ = _PROJ_FIELDS


class B2CProjGrads(ctypes.Structure):
    _fields_ = _PROJ_FIELDS


class B2CDropout(ctypes.Structure):
    _fields_ = [("p", ctypes.c_float), ("seed", ctypes.c_uint64), ("seed_dev", ctypes.c_void_p)]


B2C_OPT_MAX_SEG, B2C_OPT_MAX_CLIP, B2C_OPT_SCRATCH_BYTES = 8, 4, 16384
B2C_OPT_NSTATS = B2C_OPT_MAX_CLIP + 2


class B2COptSegment(ctypes.Structure):
    _fields_ = [("begin", ctypes.c_int64), ("end", ctypes.c_int64), ("lr_index", ctypes.c_int32), ("clip_group", ctypes.c_int32),
                ("weight_decay", ctypes.c_float)]


class B2COptHyper(ctypes.Structure):
    _fields_ = [("beta1", ctypes.c_double), ("beta2", ctypes.c_double), ("eps", ctypes.c_double), ("max_norm", ctypes.c_float), ("grad_scale", ctypes.c_float),
                ("growth_factor", ctypes.c_float), ("backoff_factor", ctypes.c_float), ("growth_interval", ctypes.c_int32)]


# every symbol include/b2c.h declares: name -> (restype, argtypes)
_vp, _i32, _i64, _f, _sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_size_t
_SHP, _PRM, _GRD, _DRP = ctypes.POINTER(B2CShape), ctypes.POINTER(B2CParams), ctypes.POINTER(B2CGrads), ctypes.POINTER(B2CDropout)
SYMBOLS = {
    "b2c_abi_version": (ctypes.c_int, []),
    "b2c_last_error": (ctypes.c_char_p, []),
    "b2c_launch_count": (ctypes.c_uint64, []),
    "b2c_workspace_bytes": (_sz, [_SHP, ctypes.c_int, ctypes.c_int]),
    "b2c_decoder_forward": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, _vp, _vp, _vp, _sz, ctypes.c_int, _DRP, _vp]),
    "b2c_decoder_prepare": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _sz, ctypes.c_int, _vp]),
    "b2c_decoder_set_initial_state": (ctypes.c_int, [_SHP, _vp, _vp, _vp, _sz, ctypes.c_int, _vp]),
    "b2c_decoder_forward_eval": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp, _sz, ctypes.c_int, _vp]),
    "b2c_decoder_forward_eval_teacher": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, ctypes.c_int, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                                        ctypes.c_int, _vp]),
    "b2c_decoder_forward_prepared": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, _vp, _vp, _vp, _sz, ctypes.c_int, _DRP, _vp]),
    "b2c_decoder_backward": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, _vp, _vp, _vp, _GRD, _vp, _vp, _sz, ctypes.c_int, _DRP, ctypes.c_int, _vp]),
    "b2c_decoder_backward_pitched": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _GRD, _vp, _vp, _sz, ctypes.c_int, _DRP, ctypes.c_int, _vp]),
    "b2c_decoder_forward_steps": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, _vp, _vp, _vp, _sz, ctypes.c_int, _DRP, _vp, _vp]),
    "b2c_decoder_forward_prepared_steps": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, _vp, _vp, _vp, _sz, ctypes.c_int, _DRP, _vp, _vp]),
    "b2c_decoder_backward_steps": (ctypes.c_int, [_SHP, _PRM, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _GRD, _vp, _vp, _sz, ctypes.c_int, _DRP, ctypes.c_int,
                                                  _vp, _vp]),
    "b2c_bump_counter": (ctypes.c_int, [_vp, _vp]),
    "b2c_debug_recur_trace": (ctypes.c_int, [_vp, _i64, _vp, _vp]),
    "b2c_join_side_work": (ctypes.c_int, [_vp]),
    "b2c_set_gemm_cta_limit": (ctypes.c_int, [ctypes.c_int32]),
    "b2c_greedy_decode": (ctypes.c_int, [_SHP, _PRM, _vp, _i64, _i64, _vp, _vp, _vp, _sz, ctypes.c_int, _vp]),
    "b2c_attention_step": (ctypes.c_int, [_SHP, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, ctypes.c_int, _vp]),
    "b2c_refinement_forward": (ctypes.c_int, [_SHP, ctypes.POINTER(B2CRefineParams), _vp, _vp, _vp, _sz, ctypes.c_int, _DRP, _vp]),
    "b2c_refinement_forward_dual": (ctypes.c_int, [_SHP, ctypes.POINTER(B2CRefineParams), _vp, _vp, _vp, _vp, _sz, ctypes.c_int, _DRP, _vp]),
    "b2c_refinement_backward": (ctypes.c_int, [_SHP, ctypes.POINTER(B2CRefineParams), _vp, _vp, ctypes.POINTER(B2CRefineGrads), _vp, _vp, _sz, ctypes.c_int, _DRP, _vp]),
    "b2c_projector_forward": (ctypes.c_int, [_SHP, ctypes.POINTER(B2CProjParams), _vp, _vp, _vp, _sz, ctypes.c_int, _DRP, _vp]),
    "b2c_projector_forward_teacher": (ctypes.c_int, [_SHP, ctypes.POINTER(B2CProjParams), _vp, ctypes.c_int, _vp, _vp, _sz, ctypes.c_int, _DRP, _vp]),
    "b2c_projector_backward": (ctypes.c_int, [_SHP, ctypes.POINTER(B2CProjParams), _vp, ctypes.POINTER(B2CProjGrads), _vp, _sz, ctypes.c_int, _DRP, _vp]),
    "b2c_count_valid": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "b2c_kd_token_loss": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _f, _f, _f, _f, _vp, _vp, _vp, _vp, ctypes.c_int, _vp]),
    "b2c_kd_token_loss_pitched": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _f, _f, _f, _f, _vp, _vp, _i64, _vp, _vp, ctypes.c_int, _vp]),
    "b2c_kd_token_loss_steps": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _f, _f, _f, _f, _vp, _vp, _i64, _vp, _vp, ctypes.c_int, _vp, _i64, _vp]),
    "b2c_kd_token_loss_teacher": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _i64, _i32, _f, _f, _f, _f, _vp, _vp, _i64, _vp, _vp, ctypes.c_int,
                                                 _vp, _i64, _vp]),
    "b2c_kd_token_eval": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _f, _vp, _vp, _vp, _vp, ctypes.c_int, _vp]),
    "b2c_kd_token_eval_teacher": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _i64, _i32, _f, _vp, _vp, _vp, _vp, ctypes.c_int, _vp]),
    "b2c_bleu1": (ctypes.c_int, [_vp, _vp, _i32, _i32, _vp, _vp]),
    "b2c_aux_loss": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _i32, _i32, _f, _f, _vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_int, _vp]),
    "b2c_aux_loss_steps": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _i32, _i32, _f, _f, _vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_int,
                                          _vp, _vp]),
    "b2c_aux_loss_teacher": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, ctypes.c_int, _i32, _i32, _i32, _f, _f, _vp, _vp, _vp, _vp, _vp,
                                            ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "b2c_loss_finalize": (ctypes.c_int, [_vp, _vp, _i64, _vp, _f, _vp, _i32, _i32, _vp, _i32, _i32, _f, _f, _f, _f, _f, _vp, _vp]),
    "b2c_loss_finalize_steps": (ctypes.c_int, [_vp, _vp, _i64, _vp, _f, _vp, _i32, _i32, _vp, _i32, _i32, _f, _f, _f, _f, _f, _vp, _vp, _vp]),
    "b2c_scale_inplace": (ctypes.c_int, [_vp, _i64, ctypes.c_int, _vp, _vp]),
    "b2c_optimizer_step": (ctypes.c_int, [_vp, _vp, _vp, _vp, ctypes.POINTER(B2COptSegment), _i32, ctypes.POINTER(B2COptHyper),
                                          _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b2c_gemm": (ctypes.c_int, [_i32, _i32, _i32, _f, _vp, _i64, ctypes.c_int, _vp, _i64, ctypes.c_int, _f, _vp, _i64, _vp,
                                ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]),
}

_lib = None


def load_library() -> ctypes.CDLL:
    """Load lib/libb2c.so (built by __graft_entry__.build()).  Fails loudly: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"b2c CUDA extension not built: {LIB_PATH} is missing. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "from the repo root (needs nvcc). There is no CPU/eager fallback for the hot path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    if lib.b2c_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libb2c.so ABI {lib.b2c_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def _check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load_library().b2c_last_error().decode("utf-8", "replace")
        exc = ValueError if rc == -1 else RuntimeError
        raise exc(f"{what} failed (code {rc}): {msg}")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name} is on {t.device}: the b2c hot path runs only on a CUDA (sm_100a) device; there is no CPU fallback")


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return B2C_F32
    if dt == torch.bfloat16:
        return B2C_BF16
    raise ValueError(f"unsupported compute dtype {dt} (use torch.float32 or torch.bfloat16)")


_TEACHER_CODES = {torch.float32: B2C_F32, torch.bfloat16: B2C_BF16, torch.float16: B2C_F16}


def teacher_operand(t: torch.Tensor, device: torch.device):
    """A teacher tensor (logits, hidden states, features for the projector) as the kernels read it -> (tensor, dtype code).
    float32, bfloat16 and float16 are read in their own precision and widened exactly in registers, so a half-precision teacher
    (autocast, or outputs cached in half precision) costs no fp32 copy; the tensor is made contiguous only if it is not.  Any other
    dtype (float64, ...) is converted to float32."""
    t = t.detach()
    code = _TEACHER_CODES.get(t.dtype)
    if code is None:
        return t.to(device=device, dtype=torch.float32).contiguous(), B2C_F32
    return t.to(device=device).contiguous(), code


def param_order(L: int) -> List[str]:
    """LSTMDecoder state_dict keys in the order DecoderFunction takes its parameter tensors."""
    names = ["embedding.weight", "attention.weight", "attention.bias", "attention_combine.weight", "attention_combine.bias"]
    for k in range(L):
        names += [f"lstm.weight_ih_l{k}", f"lstm.weight_hh_l{k}", f"lstm.bias_ih_l{k}", f"lstm.bias_hh_l{k}"]
    names += ["output_projection.0.weight", "output_projection.0.bias", "output_projection.3.weight", "output_projection.3.bias"]
    return names


def _fill_struct(st, tensors: Sequence[torch.Tensor], L: int):
    it = iter(tensors)
    st.embedding = next(it).data_ptr(); st.attn_w = next(it).data_ptr(); st.attn_b = next(it).data_ptr()
    st.comb_w = next(it).data_ptr(); st.comb_b = next(it).data_ptr()
    for k in range(L):
        st.w_ih[k] = next(it).data_ptr(); st.w_hh[k] = next(it).data_ptr()
        st.b_ih[k] = next(it).data_ptr(); st.b_hh[k] = next(it).data_ptr()
    st.out0_w = next(it).data_ptr(); st.out0_b = next(it).data_ptr(); st.out3_w = next(it).data_ptr(); st.out3_b = next(it).data_ptr()
    return st


def _master(params: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    out = []
    for p in params:
        q = p.detach()
        if q.dtype != torch.float32 or not q.is_contiguous():
            q = q.float().contiguous()
        out.append(q)
    return out


class CallOptions:
    """Per-call options of the native autograd Functions.  A module reads them from its `b2c_options` attribute at FORWARD time and
    the Function keeps them in its ctx for the backward, so nothing here is process-global: two models (or two devices, or an
    eager loop next to a GraphedKDStep) do not see each other's settings.

    grad_dest       parameter data_ptr -> fp32 tensor (a view into the flat gradient buffer of imagecaptioner_b200.ddp).  The
                    backward kernels then write that parameter's gradient straight into its slot and return the view; with
                    `.grad = None` autograd adopts it without a copy or an add kernel.  The kernels OVERWRITE, so this is only
                    for one-backward-per-step training (GraphedKDStep); leave it None when gradients are accumulated.
    defer_join      b2c_decoder_backward returns without joining its weight-gradient side branch (B2C_BWD_DEFER_JOIN); the owner
                    calls join_side_work() before the gradients are read.  Honoured only when every decoder gradient goes to a
                    grad_dest slot (a fresh tensor would be consumed by autograd's accumulation before it is written).
    after_backward  callable run right after b2c_decoder_backward is enqueued (same stream): GraphedKDStep records an event there
                    so the all-reduce of the decoder's gradient segment can start while the refinement backward still runs.
    seed_dev        int64 device tensor (1 element): the per-step dropout counter the kernels mix into the seed (B2CDropout.seed_dev),
                    so CUDA-graph replays draw fresh masks.
    background_ctas ProjectorFunction.backward only: CTA budget of its contractions when it overlaps the decoder's reverse recurrence.
    steps_dev       int32 device tensor (1 element), or None: the batch has only its first steps_dev[0] time steps (1 <= value <= T);
                    the decoder and the KD loss compute the loss and gradients of that shorter batch in their (T, B, ...) buffers, reading
                    the value at run time (the *_steps entry points of include/b2c.h), so one CUDA graph serves every caption length.
                    The caller keeps the caption / target rows past it PAD (0) and writes the value on the stream before the call."""

    def __init__(self, grad_dest=None, defer_join=False, after_backward=None, seed_dev=None, background_ctas=0, steps_dev=None):
        self.grad_dest, self.defer_join, self.after_backward, self.seed_dev = grad_dest, defer_join, after_backward, seed_dev
        self.steps_dev = steps_dev
        # > 0: the projector's backward runs as background work next to a latency-bound chain on another stream: its persistent GEMMs
        # are confined to this many CTAs (b2c_set_gemm_cta_limit) so they cannot starve the chain of SMs
        self.background_ctas = background_ctas
        self.join_pending = False      # set by DecoderFunction.backward when it deferred the join


_NO_OPTIONS = CallOptions()


def _options(opts) -> CallOptions:
    return opts if opts is not None else _NO_OPTIONS


def _dropout(p, seed, opts) -> B2CDropout:
    sd = opts.seed_dev
    return B2CDropout(float(p), int(seed), sd.data_ptr() if (sd is not None and float(p) > 0) else None)


def bump_counter(counter: torch.Tensor) -> None:
    """counter[0] += 1 on the current stream (the dropout step counter; one tiny native launch, capturable)."""
    _check(load_library().b2c_bump_counter(counter.data_ptr(), _stream()), "b2c_bump_counter")


def join_side_work() -> None:
    _check(load_library().b2c_join_side_work(_stream()), "b2c_join_side_work")


def _grad_buffers(params, master, opts=None):
    """-> (gradient tensors, all_direct): all_direct is True when every one is a registered destination slot."""
    dest = _options(opts).grad_dest
    out, all_direct = [], bool(dest)
    for p, m in zip(params, master):
        dst = dest.get(p.data_ptr()) if dest else None
        if dst is not None and dst.dtype == torch.float32 and dst.shape == m.shape and dst.is_contiguous():
            out.append(dst.view(dst.shape))      # a fresh view object: autograd adopts it as .grad only if nothing else holds it
        else:
            out.append(torch.empty_like(m))
            all_direct = False
    return out, all_direct


def workspace_bytes(shape: B2CShape, code: int, mode: int) -> int:
    lib = load_library()
    n = lib.b2c_workspace_bytes(ctypes.byref(shape), code, mode)
    if n == 0:
        _check(-1, "b2c_workspace_bytes")
    return n


class PreparedDecoder:
    """Handle of a b2c_decoder_prepare call in flight on a side stream: its workspace, and what it was prepared for."""

    def __init__(self, ws, cap, key, stream):
        self.ws, self.cap, self.key, self.stream = ws, cap, key, stream


_prepare_streams = {}


def decoder_prepare(captions: torch.Tensor, S: int, compute_dtype: torch.dtype, L: int, params: Sequence[torch.Tensor]) -> PreparedDecoder:
    """Enqueue the feature-independent part of the decoder forward (operand packing, embedding rows, layer-0 embedding gates)
    on a side stream, so that it runs underneath whatever still produces the image features on the current stream
    (AttentionRefinement).  Pass the result to DecoderFunction as `prepared`; it joins the side stream before the rest."""
    lib = load_library()
    dev = params[0].device
    if dev.type != "cuda":
        raise RuntimeError("decoder_prepare: parameters must be CUDA tensors (no CPU fallback)")
    T, B = captions.shape
    E = params[1].shape[0]
    H = params[1].shape[1] - E
    V = params[0].shape[0]
    shape = B2CShape(B, T, S, E, H, L, V)
    code = dtype_code(compute_dtype)
    cap = captions.detach().to(device=dev, dtype=torch.int64).contiguous()
    master = _master(params)
    ws = torch.empty(workspace_bytes(shape, code, B2C_WS_TRAIN), dtype=torch.uint8, device=dev)
    prm = _fill_struct(B2CParams(), master, L)
    side = _prepare_streams.get(dev.index)
    if side is None:
        side = _prepare_streams[dev.index] = torch.cuda.Stream(device=dev, priority=-1)      # needed right after the features: same rank as the main chain
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        _check(lib.b2c_decoder_prepare(ctypes.byref(shape), ctypes.byref(prm), cap.data_ptr(), ws.data_ptr(), ws.numel(), code, _stream()),
               "b2c_decoder_prepare")
    ws.record_stream(side)
    cap.record_stream(side)
    return PreparedDecoder(ws, cap, (B, T, S, E, H, L, V, code), side)


def compute_copy_of(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """`t` in the compute type, contiguous.  A tensor that a native module produced together with such a copy (RefinementFunction)
    carries it as `_b2c_compute_copy`; it is used as long as the tensor has not been modified in place since."""
    tag = getattr(t, "_b2c_compute_copy", None)
    if tag is not None:
        c, version = tag
        if c.dtype == dtype and c.shape == t.shape and c.device == t.device and t._version == version:
            return c
    return t.detach().to(dtype).contiguous()


def _pitched_rows(g: torch.Tensor, cdt: torch.dtype) -> Optional[int]:
    """Row pitch of a (T,B,V) bf16 gradient whose rows are padded to a 16-byte pitch (strides (B*ld, ld, 1), ld % 8 == 0, ld > V,
    16-byte aligned: the view KDLossFunction returns for V % 8 != 0), or None: then the gradient is made contiguous."""
    if cdt != torch.bfloat16 or g.dtype != cdt or g.dim() != 3:
        return None
    T, B, V = g.shape
    ld = g.stride(1)
    if ld <= V or ld % 8 or g.stride(2) != 1 or g.stride(0) != B * ld or g.data_ptr() % 16:
        return None
    return ld


def _steps_arg(sd: Optional[torch.Tensor]) -> Optional[int]:
    """Device pointer of a CallOptions.steps_dev tensor (validated), or None for a full-length batch."""
    if sd is None:
        return None
    if not (sd.is_cuda and sd.dtype == torch.int32 and sd.numel() == 1):
        raise ValueError(f"steps_dev must be a 1-element int32 CUDA tensor, got {sd.dtype} {tuple(sd.shape)} on {sd.device}")
    return sd.data_ptr()


class DecoderFunction(torch.autograd.Function):
    """LSTMDecoder.forward (reference src/student_model.py:205-256) as one C-ABI call each way."""

    @staticmethod
    def forward(ctx, feats, captions, compute_dtype, dropout_p, seed, L, prepared, opts, init_state, *params):
        lib = load_library()
        opts = _options(opts)
        _require_cuda(feats, "image_features")
        B, S, E = feats.shape
        T = captions.shape[0]
        H = params[1].shape[1] - E      # attention.weight is (E, H+E)
        V = params[0].shape[0]
        shape = B2CShape(B, T, S, E, H, L, V)
        code = dtype_code(compute_dtype)
        f = compute_copy_of(feats, compute_dtype)
        master = _master(params)
        if prepared is not None:
            if prepared.key != (B, T, S, E, H, L, V, code):
                raise ValueError(f"decoder was prepared for {prepared.key}, forward called with {(B, T, S, E, H, L, V, code)}")
            ws, cap = prepared.ws, prepared.cap
            torch.cuda.current_stream(feats.device).wait_stream(prepared.stream)
            fwd = "prepared"
        else:
            cap = captions.detach().to(device=feats.device, dtype=torch.int64).contiguous()
            ws = torch.empty(workspace_bytes(shape, code, B2C_WS_TRAIN), dtype=torch.uint8, device=feats.device)
            fwd = "plain"
        prm = _fill_struct(B2CParams(), master, L)
        if init_state is not None:
            # reference LSTMDecoder.forward(..., hidden=(h0, c0)): the split forward with the state written between its halves
            h0, c0 = (t.detach().to(device=feats.device, dtype=torch.float32).contiguous() for t in init_state)
            if tuple(h0.shape) != (L, B, H) or tuple(c0.shape) != (L, B, H):
                raise ValueError(f"hidden must be (h0, c0) of shape {(L, B, H)}, got {tuple(h0.shape)} and {tuple(c0.shape)}")
            if prepared is None:
                _check(lib.b2c_decoder_prepare(ctypes.byref(shape), ctypes.byref(prm), cap.data_ptr(), ws.data_ptr(), ws.numel(), code, _stream()),
                       "b2c_decoder_prepare")
            _check(lib.b2c_decoder_set_initial_state(ctypes.byref(shape), h0.data_ptr(), c0.data_ptr(), ws.data_ptr(), ws.numel(), code, _stream()),
                   "b2c_decoder_set_initial_state")
            fwd = "prepared"
        logits = torch.empty(T, B, V, dtype=compute_dtype, device=feats.device)
        hid = torch.empty(T, B, H, dtype=compute_dtype, device=feats.device)
        attw = torch.empty(T, B, S, dtype=torch.float32, device=feats.device)
        drop = _dropout(dropout_p, seed, opts)
        steps = _steps_arg(opts.steps_dev)
        args = (ctypes.byref(shape), ctypes.byref(prm), f.data_ptr(), cap.data_ptr(), logits.data_ptr(), hid.data_ptr(), attw.data_ptr(),
                ws.data_ptr(), ws.numel(), code, ctypes.byref(drop))
        if steps is None:
            _check((lib.b2c_decoder_forward if fwd == "plain" else lib.b2c_decoder_forward_prepared)(*args, _stream()), "b2c_decoder_forward")
        else:                                            # variable-length batch: the device step count of opts.steps_dev
            _check((lib.b2c_decoder_forward_steps if fwd == "plain" else lib.b2c_decoder_forward_prepared_steps)(*args, steps, _stream()),
                   "b2c_decoder_forward_steps")
        ctx.b2c = (shape, code, drop, L, ws, f, cap, master, hid, attw, feats.dtype, [p.dtype for p in params], opts, steps)
        ctx.b2c_params = params
        ctx.mark_non_differentiable(attw)
        return logits, hid, attw

    @staticmethod
    def backward(ctx, dlogits, dhid, _dattw):
        lib = load_library()
        shape, code, drop, L, ws, f, cap, master, hid, attw, feats_dtype, pdtypes, opts, steps = ctx.b2c
        cdt = f.dtype
        if dlogits is None:
            dlogits = torch.zeros(shape.T, shape.B, shape.V, dtype=cdt, device=f.device)
        ld = _pitched_rows(dlogits, cdt)
        if ld is None:
            dlogits = dlogits.to(cdt).contiguous()
        if dhid is not None:
            dhid = dhid.to(cdt).contiguous()
        grads, all_direct = _grad_buffers(ctx.b2c_params, master, opts)
        # the weight gradients are written on the library's side stream: the join may only be deferred when none of them is a
        # fresh tensor that autograd accumulates / casts on this stream right after the call returns
        defer = opts.defer_join and all_direct and all(dt == torch.float32 for dt in pdtypes)
        dfeats = torch.empty(shape.B, shape.S, shape.E, dtype=torch.float32, device=f.device)
        prm = _fill_struct(B2CParams(), master, L)
        grd = _fill_struct(B2CGrads(), grads, L)
        flags = B2C_BWD_DEFER_JOIN if defer else 0
        if steps is not None:                            # the rows past the step count of dlogits / dhid are zeros (KDLossFunction)
            _check(lib.b2c_decoder_backward_steps(ctypes.byref(shape), ctypes.byref(prm), f.data_ptr(), cap.data_ptr(), hid.data_ptr(),
                                                  attw.data_ptr(), dlogits.data_ptr(), shape.V if ld is None else ld, _ptr(dhid),
                                                  ctypes.byref(grd), dfeats.data_ptr(), ws.data_ptr(), ws.numel(), code, ctypes.byref(drop),
                                                  flags, steps, _stream()),
                   "b2c_decoder_backward_steps")
        elif ld is None:
            _check(lib.b2c_decoder_backward(ctypes.byref(shape), ctypes.byref(prm), f.data_ptr(), cap.data_ptr(), hid.data_ptr(), attw.data_ptr(),
                                            dlogits.data_ptr(), _ptr(dhid), ctypes.byref(grd), dfeats.data_ptr(), ws.data_ptr(), ws.numel(),
                                            code, ctypes.byref(drop), flags, _stream()),
                   "b2c_decoder_backward")
        else:
            _check(lib.b2c_decoder_backward_pitched(ctypes.byref(shape), ctypes.byref(prm), f.data_ptr(), cap.data_ptr(), hid.data_ptr(),
                                                    attw.data_ptr(), dlogits.data_ptr(), ld, _ptr(dhid), ctypes.byref(grd), dfeats.data_ptr(),
                                                    ws.data_ptr(), ws.numel(), code, ctypes.byref(drop), flags, _stream()),
                   "b2c_decoder_backward_pitched")
        if defer:
            opts.join_pending = True                     # the owner of `opts` calls join_side_work() and clears this
        if opts.after_backward is not None:              # GraphedKDStep: the decoder's gradients are enqueued from here on
            opts.after_backward()
        grads = [g if g.dtype == dt else g.to(dt) for g, dt in zip(grads, pdtypes)]
        dfe = dfeats if feats_dtype == torch.float32 else dfeats.to(feats_dtype)
        return (dfe, None, None, None, None, None, None, None, None, *grads)


def greedy_decode(feats: torch.Tensor, params: Sequence[torch.Tensor], L: int, max_len: int, start_id: int, end_id: int,
                  compute_dtype: torch.dtype = torch.float32):
    """Batched greedy decode on the device: returns tokens (max_len,B) int64, lengths (B) int32."""
    lib = load_library()
    _require_cuda(feats, "image_features")
    B, S, E = feats.shape
    H = params[1].shape[1] - E
    V = params[0].shape[0]
    shape = B2CShape(B, max_len, S, E, H, L, V)
    code = dtype_code(compute_dtype)
    f = feats.detach().to(compute_dtype).contiguous()
    master = _master(params)
    ws = torch.empty(workspace_bytes(shape, code, B2C_WS_DECODE), dtype=torch.uint8, device=feats.device)
    tokens = torch.empty(max_len, B, dtype=torch.int64, device=feats.device)
    lengths = torch.empty(B, dtype=torch.int32, device=feats.device)
    prm = _fill_struct(B2CParams(), master, L)
    _check(lib.b2c_greedy_decode(ctypes.byref(shape), ctypes.byref(prm), f.data_ptr(), int(start_id), int(end_id), tokens.data_ptr(),
                                 lengths.data_ptr(), ws.data_ptr(), ws.numel(), code, _stream()), "b2c_greedy_decode")
    return tokens, lengths


def attention_step(hidden: torch.Tensor, feats: torch.Tensor, attn_w: torch.Tensor, attn_b: torch.Tensor,
                   compute_dtype: torch.dtype = torch.float32):
    """LSTMDecoder.attention_mechanism as a stand-alone call: context (B,E), weights (B,S)."""
    lib = load_library()
    _require_cuda(feats, "image_features")
    B, S, E = feats.shape
    H = hidden.shape[1]
    shape = B2CShape(B, 1, S, E, H, 1, 2)
    code = dtype_code(compute_dtype)
    f = feats.detach().to(compute_dtype).contiguous()
    h = hidden.detach().to(device=feats.device, dtype=compute_dtype).contiguous()
    wa, ba = _master([attn_w, attn_b])
    ws = torch.empty(workspace_bytes(shape, code, B2C_WS_ATTN), dtype=torch.uint8, device=feats.device)
    ctx = torch.empty(B, E, dtype=compute_dtype, device=feats.device)
    wts = torch.empty(B, S, dtype=torch.float32, device=feats.device)
    _check(lib.b2c_attention_step(ctypes.byref(shape), wa.data_ptr(), ba.data_ptr(), h.data_ptr(), f.data_ptr(), ctx.data_ptr(),
                                  wts.data_ptr(), ws.data_ptr(), ws.numel(), code, _stream()), "b2c_attention_step")
    return ctx, wts


def count_valid(targets: torch.Tensor, V: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """#{0 < target < V} as an int32 device scalar (the CrossEntropyLoss(ignore_index=0) normaliser)."""
    lib = load_library()
    _require_cuda(targets, "targets")
    tg = targets.detach().to(torch.int64).contiguous()
    if out is None:
        out = torch.empty(1, dtype=torch.int32, device=targets.device)
    _check(lib.b2c_count_valid(tg.data_ptr(), tg.numel(), int(V), out.data_ptr(), _stream()), "b2c_count_valid")
    return out


class KDLossFunction(torch.autograd.Function):
    """DistillationLoss.forward (reference src/distillation_utils.py:138-200): the token pass, the fused
    feature/hidden reduction and the weighting, with all gradients produced during the forward."""

    @staticmethod
    def forward(ctx, logits, teacher_logits, targets, feats_s, feats_t, hid_s, hid_t, cfg):
        lib = load_library()
        _require_cuda(logits, "student logits")
        alpha, beta, gamma, temperature, w_ce, ce_mult, group, nval_global, unit_grad = cfg[:9]
        T, B, V = logits.shape
        # cfg[9]: CallOptions.steps_dev -- a variable-length batch of the first steps_dev[0] of T steps (its targets past them are PAD)
        steps = _steps_arg(cfg[9] if len(cfg) > 9 else None)
        N = T * B
        dev = logits.device
        cdt = logits.dtype if logits.dtype in (torch.float32, torch.bfloat16) else torch.float32
        code = dtype_code(cdt)
        y = logits.detach().to(cdt).contiguous()
        z, zcode = teacher_operand(teacher_logits, dev)
        tg = targets.detach().to(device=dev, dtype=torch.int64).contiguous()
        st = _stream()
        if nval_global is not None:                # the caller already holds the (global) non-PAD count on the device
            nval = nval_global
        else:
            nval = count_valid(tg, V)
            if group is not None:                  # data parallel: the CE normaliser is the GLOBAL non-PAD count
                torch.distributed.all_reduce(nval, group=group)
        rows = torch.empty(2, N, dtype=torch.float32, device=dev)
        if cdt == torch.bfloat16 and V % 8 != 0:
            # the logits gradient lives at row pitch Vp = roundup(V, 8) (columns V..Vp-1 written as zeros) and leaves as the (T,B,V)
            # view: DecoderFunction.backward hands the pitch on, and the vocabulary head's backward contractions stay on tensor cores
            Vp = (V + 7) // 8 * 8
            dlogits_buf = torch.empty(T, B, Vp, dtype=cdt, device=dev)
            dlogits = dlogits_buf[..., :V]
        else:
            Vp = V
            dlogits = dlogits_buf = torch.empty_like(y)
        # steps (variable-length batch): rows past the step count get zero losses and gradients; Vp != V: pitched dlogits
        _check(lib.b2c_kd_token_loss_teacher(y.data_ptr(), z.data_ptr(), zcode, tg.data_ptr(), N, V, float(temperature), float(alpha),
                                             float(w_ce), float(ce_mult), nval.data_ptr(), dlogits_buf.data_ptr(), Vp, rows[0].data_ptr(),
                                             rows[1].data_ptr(), code, steps, B, st), "b2c_kd_token_loss_teacher")
        fs = ft = hs = ht = dfs = dft = dhs = feat_part = hid_part = None
        Ss = St = E = H = Th = 0
        fcode, hcode = code, B2C_F32
        if feats_s is not None and feats_t is not None:
            # fp32 student features stay fp32 (the reference's encoder features reach the loss un-cast); otherwise the compute type
            fs = feats_s.detach().contiguous() if feats_s.dtype == torch.float32 else feats_s.detach().to(cdt).contiguous()
            fcode = dtype_code(fs.dtype)
            ft = feats_t.detach().to(device=dev, dtype=torch.float32).contiguous()
            _, Ss, E = fs.shape
            St = ft.shape[1]
            dfs = torch.empty(B, Ss, E, dtype=torch.float32, device=dev)
            dft = torch.empty(B, St, E, dtype=torch.float32, device=dev)
            feat_part = torch.empty(B, 2, dtype=torch.float32, device=dev)
        if hid_s is not None and hid_t is not None:
            hs = hid_s.detach().to(cdt).contiguous()
            ht, hcode = teacher_operand(hid_t, dev)
            Th, H = ht.shape[0], ht.shape[2]
            dhs = torch.empty_like(hs)
            hid_part = torch.empty(Th * B, 2, dtype=torch.float32, device=dev)
        if fs is not None or hs is not None:
            _check(lib.b2c_aux_loss_teacher(_ptr(fs), _ptr(ft), B, Ss, St, E, _ptr(hs), _ptr(ht), hcode, hs.shape[0] if hs is not None else 0,
                                            Th, H, float(beta), float(gamma), _ptr(dfs), _ptr(dft), _ptr(dhs), _ptr(feat_part), _ptr(hid_part),
                                            code, fcode, steps, st), "b2c_aux_loss_teacher")
        out5 = torch.empty(5, dtype=torch.float32, device=dev)
        fin = (rows[0].data_ptr(), rows[1].data_ptr(), N, nval.data_ptr(), float(ce_mult), _ptr(feat_part), B, E,
               _ptr(hid_part), Th, H, float(temperature), float(alpha), float(beta), float(gamma), float(w_ce), out5.data_ptr())
        if steps is None:
            _check(lib.b2c_loss_finalize(*fin, st), "b2c_loss_finalize")
        else:
            _check(lib.b2c_loss_finalize_steps(*fin, steps, st), "b2c_loss_finalize_steps")
        ctx.b2c = dict(dlogits=dlogits, dlogits_buf=dlogits_buf, dfs=dfs, dft=dft, dhs=dhs, code=code, used=False, unit_grad=bool(unit_grad),
                       dtypes=(logits.dtype, None if feats_s is None else feats_s.dtype,
                               None if feats_t is None else feats_t.dtype, None if hid_s is None else hid_s.dtype))
        ctx.mark_non_differentiable(out5)
        return out5[0].clone(), out5

    @staticmethod
    def backward(ctx, grad_loss, _g5):
        lib = load_library()
        sv = ctx.b2c
        if sv["used"]:
            raise RuntimeError("KDLossFunction.backward ran twice: its gradients are scaled in place (retain_graph is not supported)")
        sv["used"] = True
        if not sv["unit_grad"]:          # unit_grad: the caller guarantees loss.backward() with grad_output == 1 (GraphedKDStep)
            scale = grad_loss.detach().to(torch.float32).reshape(1).contiguous()
            st = _stream()
            # the whole padded buffer: its padding columns are zeros and stay zeros
            for key, code in (("dlogits_buf", sv["code"]), ("dfs", B2C_F32), ("dft", B2C_F32), ("dhs", sv["code"])):
                t = sv[key]
                if t is not None:
                    _check(lib.b2c_scale_inplace(t.data_ptr(), t.numel(), code, scale.data_ptr(), st), "b2c_scale_inplace")
        dt_l, dt_fs, dt_ft, dt_hs = sv["dtypes"]

        def cast(t, dt):
            return None if t is None else (t if t.dtype == dt else t.to(dt))

        return cast(sv["dlogits"], dt_l), None, None, cast(sv["dfs"], dt_fs), cast(sv["dft"], dt_ft), cast(sv["dhs"], dt_hs), None, None


def _eval_finish(rows, nval, B, feats_s, feats_t, hid_s, hid_t, alpha, beta, gamma, temperature, w_ce, ce_mult, cdt, code, dev):
    """feature / hidden KD without gradients + the fixed-order finalize on per-row token partials -> out5 (device)."""
    lib = load_library()
    st = _stream()
    N = rows.shape[1]
    fs = ft = hs = ht = feat_part = hid_part = None
    Ss = St = E = H = Th = 0
    fcode, hcode = code, B2C_F32
    if feats_s is not None and feats_t is not None:
        fs = feats_s.detach().contiguous() if feats_s.dtype == torch.float32 else feats_s.detach().to(cdt).contiguous()
        fcode = dtype_code(fs.dtype)
        ft = feats_t.detach().to(device=dev, dtype=torch.float32).contiguous()
        _, Ss, E = fs.shape
        St = ft.shape[1]
        feat_part = torch.empty(B, 2, dtype=torch.float32, device=dev)
    if hid_s is not None and hid_t is not None:
        hs = hid_s.detach().to(cdt).contiguous()
        ht, hcode = teacher_operand(hid_t, dev)
        Th, H = ht.shape[0], ht.shape[2]
        hid_part = torch.empty(Th * B, 2, dtype=torch.float32, device=dev)
    if fs is not None or hs is not None:
        _check(lib.b2c_aux_loss_teacher(_ptr(fs), _ptr(ft), B, Ss, St, E, _ptr(hs), _ptr(ht), hcode, hs.shape[0] if hs is not None else 0, Th, H,
                                        float(beta), float(gamma), None, None, None, _ptr(feat_part), _ptr(hid_part), code, fcode, None, st),
               "b2c_aux_loss_teacher")
    out5 = torch.empty(5, dtype=torch.float32, device=dev)
    _check(lib.b2c_loss_finalize(rows[0].data_ptr(), rows[1].data_ptr(), N, nval.data_ptr(), float(ce_mult), _ptr(feat_part), B, E,
                                 _ptr(hid_part), Th, H, float(temperature), float(alpha), float(beta), float(gamma), float(w_ce),
                                 out5.data_ptr(), st), "b2c_loss_finalize")
    return out5


@torch.no_grad()
def kd_eval(logits, teacher_logits, targets, feats_s, feats_t, hid_s, hid_t, alpha, beta, gamma, temperature, w_ce, nval_global=None,
            ce_mult=1.0):
    """DistillationLoss without gradients (validate_student_model): -> (out5 device tensor [total, ce, token_kd, feature_kd,
    hidden_kd], predicted tokens (T,B) int32 = logits.argmax(-1), taken in the same pass over the logits)."""
    lib = load_library()
    _require_cuda(logits, "student logits")
    T, B, V = logits.shape
    N, dev = T * B, logits.device
    cdt = logits.dtype if logits.dtype in (torch.float32, torch.bfloat16) else torch.float32
    code = dtype_code(cdt)
    y = logits.detach().to(cdt).contiguous()
    z, zcode = teacher_operand(teacher_logits, dev)
    tg = targets.detach().to(device=dev, dtype=torch.int64).contiguous()
    nval = nval_global if nval_global is not None else count_valid(tg, V)
    rows = torch.empty(2, N, dtype=torch.float32, device=dev)
    pred = torch.empty(T, B, dtype=torch.int32, device=dev)
    _check(lib.b2c_kd_token_eval_teacher(y.data_ptr(), z.data_ptr(), zcode, tg.data_ptr(), N, V, float(temperature), nval.data_ptr(),
                                         rows[0].data_ptr(), rows[1].data_ptr(), pred.data_ptr(), code, _stream()), "b2c_kd_token_eval_teacher")
    out5 = _eval_finish(rows, nval, B, feats_s, feats_t, hid_s, hid_t, alpha, beta, gamma, temperature, w_ce, ce_mult, cdt, code, dev)
    return out5, pred


@torch.no_grad()
def decoder_forward_eval(feats: torch.Tensor, captions: torch.Tensor, teacher_logits: torch.Tensor, targets: torch.Tensor,
                         temperature: float, L: int, params: Sequence[torch.Tensor]):
    """Teacher-forced decoder forward for validation WITHOUT the logits tensor (b2c_decoder_forward_eval, bf16 mode): ->
    hidden_top (T,B,H) bf16, attention weights (T,B,S) fp32, rows (2, T*B) fp32 = per-row [KL, CE] partials, predicted tokens (T,B)."""
    lib = load_library()
    _require_cuda(feats, "image_features")
    B, S, E = feats.shape
    T = captions.shape[0]
    H = params[1].shape[1] - E
    V = params[0].shape[0]
    dev = feats.device
    shape = B2CShape(B, T, S, E, H, L, V)
    code = B2C_BF16
    f = feats.detach().to(torch.bfloat16).contiguous()
    cap = captions.detach().to(device=dev, dtype=torch.int64).contiguous()
    z, zcode = teacher_operand(teacher_logits, dev)
    tg = targets.detach().to(device=dev, dtype=torch.int64).contiguous()
    if tuple(z.shape) != (T, B, V) or tuple(tg.shape) != (T, B):
        raise ValueError(f"teacher logits {tuple(z.shape)} / targets {tuple(tg.shape)} do not match (T,B,V) = {(T, B, V)}")
    master = _master(params)
    ws = torch.empty(workspace_bytes(shape, code, B2C_WS_TRAIN), dtype=torch.uint8, device=dev)
    hid = torch.empty(T, B, H, dtype=torch.bfloat16, device=dev)
    attw = torch.empty(T, B, S, dtype=torch.float32, device=dev)
    rows = torch.empty(2, T * B, dtype=torch.float32, device=dev)
    pred = torch.empty(T, B, dtype=torch.int32, device=dev)
    prm = _fill_struct(B2CParams(), master, L)
    _check(lib.b2c_decoder_forward_eval_teacher(ctypes.byref(shape), ctypes.byref(prm), f.data_ptr(), cap.data_ptr(), z.data_ptr(), zcode,
                                                tg.data_ptr(), float(temperature), hid.data_ptr(), attw.data_ptr(), rows[0].data_ptr(),
                                                rows[1].data_ptr(), pred.data_ptr(), ws.data_ptr(), ws.numel(), code, _stream()),
           "b2c_decoder_forward_eval_teacher")
    return hid, attw, rows, pred


@torch.no_grad()
def kd_eval_rows(rows, pred, targets, V, feats_s, feats_t, hid_s, hid_t, alpha, beta, gamma, temperature, w_ce, nval_global=None, ce_mult=1.0):
    """The rest of the validation loss on per-row token partials that came out of decoder_forward_eval: -> (out5, pred)."""
    dev = rows.device
    tg = targets.detach().to(device=dev, dtype=torch.int64).contiguous()
    nval = nval_global if nval_global is not None else count_valid(tg, V)
    out5 = _eval_finish(rows, nval, tg.shape[1], feats_s, feats_t, hid_s, hid_t, alpha, beta, gamma, temperature, w_ce, ce_mult,
                        torch.bfloat16, B2C_BF16, dev)
    return out5, pred


@torch.no_grad()
def bleu1(predicted: torch.Tensor, targets: torch.Tensor) -> torch.Tensor:
    """compute_bleu_score for every sample: predicted (T,B) int32/int64, targets (T,B) -> (B) fp32 on the device."""
    lib = load_library()
    _require_cuda(predicted, "predicted tokens")
    T, B = predicted.shape
    p = predicted.detach().to(torch.int32).contiguous()
    t = targets.detach().to(device=p.device, dtype=torch.int64).contiguous()
    out = torch.empty(B, dtype=torch.float32, device=p.device)
    _check(lib.b2c_bleu1(p.data_ptr(), t.data_ptr(), T, B, out.data_ptr(), _stream()), "b2c_bleu1")
    return out


REFINE_PARAM_ORDER = ["attention.in_proj_weight", "attention.in_proj_bias", "attention.out_proj.weight", "attention.out_proj.bias",
                      "ffn.0.weight", "ffn.0.bias", "ffn.3.weight", "ffn.3.bias", "norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"]
PROJ_PARAM_ORDER = ["feature_projection.0.weight", "feature_projection.0.bias", "feature_projection.3.weight", "feature_projection.3.bias"]


def _fill_flat(st, tensors):
    for (name, _), t in zip(st._fields_, tensors):
        setattr(st, name, t.data_ptr())
    return st


class RefinementFunction(torch.autograd.Function):
    """AttentionRefinement.forward (reference src/student_model.py:72-118): QKV / out-proj / FFN contractions on the tcgen05
    GEMM, the 49x49 4-head attention core, residual LayerNorms and every gradient in native kernels."""

    @staticmethod
    def forward(ctx, x, compute_dtype, dropout_p, seed, heads, opts, *params):
        lib = load_library()
        opts = _options(opts)
        _require_cuda(x, "features")
        B, S, E = x.shape
        shape = B2CShape(B, 1, S, E, heads, 1, 2)
        code = dtype_code(compute_dtype)
        xf = x.detach().to(torch.float32).contiguous()
        master = _master(params)
        ws = torch.empty(workspace_bytes(shape, code, B2C_WS_REFINE), dtype=torch.uint8, device=x.device)
        out = torch.empty(B, S, E, dtype=torch.float32, device=x.device)      # fp32 residual stream in both modes
        prm = _fill_flat(B2CRefineParams(), master)
        drop = _dropout(dropout_p, seed, opts)
        # bf16 mode: the final LayerNorm also leaves the features in the compute type; the decoder picks that copy up (compute_copy_of)
        # instead of casting the fp32 output again (one element-wise pass less between the two modules, on the critical path)
        out_c = torch.empty(B, S, E, dtype=compute_dtype, device=x.device) if compute_dtype != torch.float32 else None
        _check(lib.b2c_refinement_forward_dual(ctypes.byref(shape), ctypes.byref(prm), xf.data_ptr(), out.data_ptr(), _ptr(out_c), ws.data_ptr(),
                                               ws.numel(), code, ctypes.byref(drop), _stream()), "b2c_refinement_forward_dual")
        ctx.b2c = (shape, code, drop, ws, master, x.dtype, [p.dtype for p in params], xf, opts)
        ctx.b2c_params = params
        if out_c is not None:
            out._b2c_compute_copy = (out_c, out._version)
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = load_library()
        shape, code, drop, ws, master, x_dtype, pdtypes, xf, opts = ctx.b2c
        dout = dout.to(torch.float32).contiguous()
        grads, _ = _grad_buffers(ctx.b2c_params, master, opts)
        dx = torch.empty(shape.B, shape.S, shape.E, dtype=torch.float32, device=dout.device)
        prm = _fill_flat(B2CRefineParams(), master)
        grd = _fill_flat(B2CRefineGrads(), grads)
        _check(lib.b2c_refinement_backward(ctypes.byref(shape), ctypes.byref(prm), xf.data_ptr(), dout.data_ptr(), ctypes.byref(grd), dx.data_ptr(),
                                           ws.data_ptr(), ws.numel(), code, ctypes.byref(drop), _stream()), "b2c_refinement_backward")
        grads = [g if g.dtype == dt else g.to(dt) for g, dt in zip(grads, pdtypes)]
        return (dx if x_dtype == torch.float32 else dx.to(x_dtype), None, None, None, None, None, *grads)


class ProjectorFunction(torch.autograd.Function):
    """FeatureProjector.forward (reference src/distillation_utils.py:233-252): Linear+ReLU(+dropout) on the tcgen05 GEMM, LayerNorm,
    token pooling, and the parameter gradients, in native kernels.  `params` is empty for the identity channel projection."""

    @staticmethod
    def forward(ctx, x, compute_dtype, dropout_p, seed, out_tokens, student_dim, opts, *params):
        lib = load_library()
        opts = _options(opts)
        _require_cuda(x, "teacher features")
        B, St, Et = x.shape
        shape = B2CShape(B, out_tokens, St, Et, student_dim, 1, 2)
        code = dtype_code(compute_dtype)
        xt, xcode = teacher_operand(x, x.device)
        master = _master(params)
        prm = _fill_flat(B2CProjParams(), master) if master else B2CProjParams()
        nbytes = workspace_bytes(shape, code, B2C_WS_PROJ) if master else 256
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        out = torch.empty(B, out_tokens, student_dim, dtype=torch.float32, device=x.device)
        drop = _dropout(dropout_p, seed, opts)
        _check(lib.b2c_projector_forward_teacher(ctypes.byref(shape), ctypes.byref(prm), xt.data_ptr(), xcode, out.data_ptr(), ws.data_ptr(),
                                                 ws.numel(), code, ctypes.byref(drop), _stream()), "b2c_projector_forward_teacher")
        ctx.b2c = (shape, code, drop, ws, master, [p.dtype for p in params], opts)
        ctx.b2c_params = params
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = load_library()
        shape, code, drop, ws, master, pdtypes, opts = ctx.b2c
        if not master:
            return (None,) * 7
        dout = dout.to(torch.float32).contiguous()
        grads, _ = _grad_buffers(ctx.b2c_params, master, opts)
        prm = _fill_flat(B2CProjParams(), master)
        grd = _fill_flat(B2CProjGrads(), grads)
        bg = int(getattr(opts, "background_ctas", 0) or 0)
        if bg > 0:
            _check(lib.b2c_set_gemm_cta_limit(bg), "b2c_set_gemm_cta_limit")
        try:
            _check(lib.b2c_projector_backward(ctypes.byref(shape), ctypes.byref(prm), dout.data_ptr(), ctypes.byref(grd), ws.data_ptr(), ws.numel(),
                                              code, ctypes.byref(drop), _stream()), "b2c_projector_backward")
        finally:
            if bg > 0:
                lib.b2c_set_gemm_cta_limit(0)
        grads = [g if g.dtype == dt else g.to(dt) for g, dt in zip(grads, pdtypes)]
        return (None, None, None, None, None, None, None, *grads)


def gemm(A: torch.Tensor, Bm: torch.Tensor, M: int, N: int, K: int, a_mn: bool = False, b_mn: bool = False,
         out_dtype: torch.dtype = torch.float32, bias: Optional[torch.Tensor] = None, relu: bool = False,
         alpha: float = 1.0, beta: float = 0.0, C: Optional[torch.Tensor] = None, impl: int = 0,
         lda: Optional[int] = None, ldb: Optional[int] = None) -> torch.Tensor:
    """Test hook for the contraction tiles (tcgen05 for bf16 operands, FFMA for fp32)."""
    lib = load_library()
    _require_cuda(A, "A")
    lda = lda if lda is not None else A.stride(0)
    ldb = ldb if ldb is not None else Bm.stride(0)
    if C is None:
        C = torch.zeros(M, N, dtype=out_dtype, device=A.device)
    _check(lib.b2c_gemm(M, N, K, float(alpha), A.data_ptr(), lda, int(a_mn), Bm.data_ptr(), ldb, int(b_mn), float(beta), C.data_ptr(),
                        C.stride(0), _ptr(bias), int(relu), dtype_code(A.dtype), dtype_code(C.dtype), impl, _stream()), "b2c_gemm")
    return C
