"""The training loss on the GPU — the reference's ``PPNLoss`` (main.py:125-216) as two fused kernels.

``ppn_loss_forward`` reads the head tensor and the ten encoded targets once and writes the five batch-mean terms;
``ppn_loss_backward`` reads them once more and writes the gradient of the head tensor, every element once.
Nothing head-sized is kept between the two: the autograd graph holds references to the inputs only.

    enc = TargetEncoder(cfg)
    criterion = PPNLoss(cfg)
    batch = enc.encode(samples)
    out = model(images)                                                  # [B, C, H, W] fp32
    terms = criterion(out, batch.delta, batch.weight, batch.weight_ij, batch.tx_half, batch.ty_half,
                      batch.tx, batch.ty, batch.tw, batch.th, batch.te)
    loss = sum(l * t for l, t in zip(lambdas, terms))                    # the reference weights by GradNorm
    loss.backward()

Under mixed precision (the reference trains under apex AMP, main.py:282-289) the head may be fp16 or bf16, and te /
weight_ij may be stored in the head's type (``TargetEncoder(cfg, limb_dtype=...)``): the loss is the fp32 loss on
the exactly widened inputs and the gradient comes back in the head's type, rounded once — no fp32 copy of the head.

``PPNLoss(cfg, from_logits=True)`` takes the conv output before the model's final sigmoid, as ``BCEWithLogitsLoss``
does: the kernels apply the sigmoid as they load each element and its derivative as they store each gradient, so
the sigmoid's own pass over the head and autograd's sigmoid backward never run.  :func:`sigmoid` is that sigmoid
alone (fp32 out), for parsing the output of a model trained that way.

The reference's training loop is not part of this project: the loss is specified by the float64 restatement
described in DESIGN.md §11 (IoU differentiable in x, y, w, h; eps = 1e-6 in the IoU denominator; L_resp
unweighted), not by bit parity with main.py.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .config import PPNConfig
from .parser import _CConfig

# the criterion's argument order (main.py's call site) — NOT the order of TargetBatch.as_list(), which follows
# __getitem__ (tx, ty, tx_half, ty_half)
ARG_ORDER = ("delta", "weight", "weight_ij", "tx_half", "ty_half", "tx", "ty", "tw", "th", "te")
TERMS = ("loss_resp", "loss_iou", "loss_coor", "loss_size", "loss_limb")
HEAD_DTYPES = {torch.float32: _lib.HEAD_F32, torch.float16: _lib.HEAD_F16, torch.bfloat16: _lib.HEAD_BF16}


class _PPNLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, crit, feature_map, *targets):
        loss = crit._launch_forward(feature_map, targets, torch.empty(5, dtype=torch.float32, device=feature_map.device))
        ctx.crit = crit
        ctx.save_for_backward(feature_map, *targets)
        ctx.set_materialize_grads(False)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        if grad_loss is None or not ctx.needs_input_grad[1]:          # no term reaches the loss: nothing to launch
            return (None,) * (2 + len(ARG_ORDER))
        feature_map, *targets = ctx.saved_tensors
        grad = ctx.crit._launch_backward(feature_map, targets, grad_loss.to(torch.float32).contiguous(),
                                         torch.empty_like(feature_map))
        return (None, grad) + (None,) * len(ARG_ORDER)


def sigmoid(x: torch.Tensor) -> torch.Tensor:
    """1 / (1 + exp(-x)) of a float32 / float16 / bfloat16 CUDA tensor, as a new float32 tensor of the same shape:
    the exact values ``PPNLoss(cfg, from_logits=True)`` computes from logits (ppn_sigmoid), e.g. the head tensor that
    :class:`parser.PoseParser` reads from a model trained on logits.  A 16-bit input is widened exactly; the result is
    not rounded back to it.  Runs on the current stream of x's device."""
    if not isinstance(x, torch.Tensor) or x.dtype not in HEAD_DTYPES or x.device.type != "cuda":
        raise ValueError(f"sigmoid takes a float32, float16 or bfloat16 CUDA tensor, got "
                         f"{(x.dtype, x.device) if isinstance(x, torch.Tensor) else type(x)}")
    x = x.contiguous()
    y = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().ppn_sigmoid(x.data_ptr(), HEAD_DTYPES[x.dtype], y.data_ptr(), x.numel(),
                                          C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)), "ppn_sigmoid")
    return y


class PPNLoss(torch.nn.Module):
    """``criterion(feature_map, delta, weight, weight_ij, tx_half, ty_half, tx, ty, tw, th, te)`` ->
    ``(loss_resp, loss_iou, loss_coor, loss_size, loss_limb)``, five 0-dim fp32 tensors on the head's device.

    The arguments come in the reference criterion's order: ``tx_half, ty_half`` BEFORE ``tx, ty``.  That is not
    the order of :meth:`dataset.TargetBatch.as_list` (``tx, ty, tx_half, ty_half``, as ``__getitem__`` returns
    them): pass the targets by name, as in the module docstring, or through :meth:`from_batch`.

    feature_map: [B, 6K + E*sH*sW, H, W] fp32, fp16 or bf16, contiguous, on a CUDA device — the sigmoid output the
    reference's model returns; the eight small targets [B, K, H, W] fp32; weight_ij and te [B, E, sH, sW, H, W],
    both fp32 or both in the dtype of a 16-bit feature_map; all contiguous, on the same device.  Anything else
    raises ValueError.  A 16-bit feature_map gets its gradient in its own dtype: the fp32 gradient of the widened
    inputs, rounded once to nearest even (overflow to +-inf, which a GradScaler detects).  The gradient flows into ``feature_map``
    only.  Terms that do not reach the final loss get no upstream gradient and are skipped in the backward; the
    upstream gradients never travel to the host.

    from_logits: feature_map (in every method) is the conv output BEFORE the model's sigmoid, and every channel goes
    through s = :func:`sigmoid` (in fp32, also for a 16-bit feature_map) before the loss above is applied to s.  The
    gradient is that of the logits: the fp32 gradient of s times (1 - s) times s, rounded once to feature_map's
    dtype.  Types, shapes and checks are the same.
    """

    def __init__(self, cfg: PPNConfig, device=None, from_logits: bool = False):
        super().__init__()
        self.from_logits = bool(from_logits)
        if not torch.cuda.is_available():
            raise RuntimeError("PPNLoss needs a CUDA device: there is no CPU path")
        self.cfg = cfg
        dev = torch.device("cuda" if device is None else device)
        if dev.type != "cuda":
            raise ValueError(f"PPNLoss runs on a CUDA device, not {dev}")
        # "cuda" without an index means the current device; tensors always carry their index
        self.device = torch.device("cuda", torch.cuda.current_device() if dev.index is None else dev.index)
        self.lib = _lib.lib()
        self.c = _CConfig(cfg)
        self._shapes = {}             # (B, head dtype code) -> PPNShape
        self._ws = None
        self._ws_need = {}            # B -> workspace bytes (ppn_loss_workspace_bytes is pure arithmetic)

    # ---- plumbing ------------------------------------------------------------------------------------------- #
    def _guard(self):
        return torch.cuda.device(self.device)

    def _stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _shape(self, B: int, head_dtype: int = _lib.HEAD_F32) -> _lib.PPNShape:
        s = self._shapes.get((B, head_dtype))
        if s is None:
            s = self._shapes[(B, head_dtype)] = self.c.shape(B, head_dtype)
        return s

    def _workspace(self, B: int) -> torch.Tensor:
        need = self._ws_need.get(B)
        if need is None:
            n = C.c_size_t()
            _lib.check(self.lib.ppn_loss_workspace_bytes(C.byref(self._shape(B)), C.byref(n)), "ppn_loss_workspace_bytes")
            need = self._ws_need[B] = n.value
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 256), dtype=torch.uint8, device=self.device)
        return self._ws

    @staticmethod
    def _targets_struct(targets) -> _lib.PPNTargets:
        by_name = dict(zip(ARG_ORDER, targets))
        return _lib.PPNTargets(*[by_name[n].data_ptr() for n in _lib.TARGET_NAMES])

    def _check(self, feature_map, targets) -> int:
        """Raises ValueError unless the call is one the kernels take; returns B."""
        cfg = self.cfg
        if len(targets) != len(ARG_ORDER):
            raise ValueError(f"expected the {len(ARG_ORDER)} targets {ARG_ORDER}, got {len(targets)}")
        if not isinstance(feature_map, torch.Tensor) or feature_map.dim() != 4 or \
                tuple(feature_map.shape[1:]) != (cfg.C, cfg.H, cfg.W):
            raise ValueError(f"feature_map must be [B, {cfg.C}, {cfg.H}, {cfg.W}], got "
                             f"{tuple(feature_map.shape) if isinstance(feature_map, torch.Tensor) else type(feature_map)}")
        B = feature_map.shape[0]
        if B < 1:
            raise ValueError("the batch mean needs at least one image")
        small = (B, cfg.K, cfg.H, cfg.W)
        big = (B, cfg.E, cfg.sH, cfg.sW, cfg.H, cfg.W)
        if feature_map.dtype not in HEAD_DTYPES:
            raise ValueError(f"feature_map must be float32, float16 or bfloat16, got {feature_map.dtype}")
        limb = dict(zip(ARG_ORDER, targets))["te"]
        limb_dtype = limb.dtype if isinstance(limb, torch.Tensor) else None
        limb_ok = (torch.float32, feature_map.dtype)          # the limb targets: fp32 or the head's 16-bit type
        for name, t in (("feature_map", feature_map),) + tuple(zip(ARG_ORDER, targets)):
            want = big if name in ("weight_ij", "te") else (feature_map.shape if name == "feature_map" else small)
            if not isinstance(t, torch.Tensor):
                raise ValueError(f"{name} must be a tensor, got {type(t)}")
            if name in ("weight_ij", "te"):
                if t.dtype not in limb_ok or t.dtype != limb_dtype:
                    raise ValueError(f"weight_ij and te must both be float32 or both {feature_map.dtype}, got {t.dtype} "
                                     f"(te {limb_dtype})")
            elif name != "feature_map" and t.dtype != torch.float32:
                raise ValueError(f"{name} must be float32, got {t.dtype}")
            if tuple(t.shape) != tuple(want):
                raise ValueError(f"{name} must have shape {tuple(want)}, got {tuple(t.shape)}")
            if t.device != self.device:
                raise ValueError(f"{name} is on {t.device}, the loss on {self.device}")
            if not t.is_contiguous():
                raise ValueError(f"{name} must be contiguous")
        return B

    # ---- the criterion ---------------------------------------------------------------------------------------- #
    def forward(self, feature_map, delta, weight, weight_ij, tx_half, ty_half, tx, ty, tw, th, te):
        targets = (delta, weight, weight_ij, tx_half, ty_half, tx, ty, tw, th, te)
        self._check(feature_map, targets)
        targets = tuple(t.detach() for t in targets)          # the targets get no gradient
        loss = _PPNLossFunction.apply(self, feature_map, *targets)
        return tuple(loss.unbind(0))

    def from_batch(self, feature_map, batch):
        """The same call with the targets taken by name from a :class:`dataset.TargetBatch`."""
        return self(feature_map, *[getattr(batch, n) for n in ARG_ORDER])

    def forward_raw(self, feature_map, *targets) -> torch.Tensor:
        """The forward export without autograd: loss[5] fp32 on the device (targets in the criterion's order)."""
        self._check(feature_map, targets)
        return self._launch_forward(feature_map, targets, torch.empty(5, dtype=torch.float32, device=self.device))

    def backward_raw(self, feature_map, *targets, grad_loss: torch.Tensor, out=None) -> torch.Tensor:
        """The backward export without autograd: sum_t grad_loss[t] * dL_t/d(feature_map), grad_loss fp32 [5] on
        the device; written into `out` (like feature_map, in its dtype) when given."""
        self._check(feature_map, targets)
        if grad_loss.dtype != torch.float32 or tuple(grad_loss.shape) != (5,) or grad_loss.device != self.device:
            raise ValueError("grad_loss must be a float32 [5] tensor on the loss's device")
        if out is None:
            out = torch.empty_like(feature_map)
        elif out.dtype != feature_map.dtype or out.shape != feature_map.shape or out.device != self.device or \
                not out.is_contiguous():
            raise ValueError(f"out must be a contiguous {feature_map.dtype} tensor like feature_map")
        return self._launch_backward(feature_map, targets, grad_loss.contiguous(), out)

    @staticmethod
    def _options(feature_map, targets):
        """None for an fp32 head (the fp32 exports), else the (shape dtype code, PPNLossOptions) of the _opt exports."""
        if feature_map.dtype == torch.float32:
            return None
        te = targets[ARG_ORDER.index("te")]
        return HEAD_DTYPES[feature_map.dtype], _lib.PPNLossOptions(HEAD_DTYPES[te.dtype])

    def _logits_options(self, feature_map, targets):
        """(shape dtype code, PPNLossOptions) of the _logits exports, which take every dtype pair."""
        te = targets[ARG_ORDER.index("te")]
        return HEAD_DTYPES[feature_map.dtype], _lib.PPNLossOptions(HEAD_DTYPES[te.dtype])

    def _launch_forward(self, feature_map, targets, loss):
        B = feature_map.shape[0]
        ws = self._workspace(B)                 # the same for every dtype (ppn_loss_workspace_bytes_opt)
        tg = self._targets_struct(targets)
        if self.from_logits:
            code, opt = self._logits_options(feature_map, targets)
            with self._guard():
                _lib.check(self.lib.ppn_loss_forward_logits(feature_map.data_ptr(), C.byref(self._shape(B, code)), C.byref(tg),
                                                            C.byref(opt), loss.data_ptr(), ws.data_ptr(), ws.numel(),
                                                            self._stream()),
                           "ppn_loss_forward_logits")
            return loss
        opt = self._options(feature_map, targets)
        with self._guard():
            if opt is None:
                _lib.check(self.lib.ppn_loss_forward(feature_map.data_ptr(), C.byref(self._shape(B)), C.byref(tg),
                                                     loss.data_ptr(), ws.data_ptr(), ws.numel(), self._stream()),
                           "ppn_loss_forward")
            else:
                _lib.check(self.lib.ppn_loss_forward_opt(feature_map.data_ptr(), C.byref(self._shape(B, opt[0])), C.byref(tg),
                                                         C.byref(opt[1]), loss.data_ptr(), ws.data_ptr(), ws.numel(),
                                                         self._stream()),
                           "ppn_loss_forward_opt")
        return loss

    def _launch_backward(self, feature_map, targets, grad_loss, grad_head):
        B = feature_map.shape[0]
        tg = self._targets_struct(targets)
        if self.from_logits:
            code, opt = self._logits_options(feature_map, targets)
            with self._guard():
                _lib.check(self.lib.ppn_loss_backward_logits(feature_map.data_ptr(), C.byref(self._shape(B, code)), C.byref(tg),
                                                             C.byref(opt), grad_loss.data_ptr(), grad_head.data_ptr(),
                                                             self._stream()),
                           "ppn_loss_backward_logits")
            return grad_head
        opt = self._options(feature_map, targets)
        with self._guard():
            if opt is None:
                _lib.check(self.lib.ppn_loss_backward(feature_map.data_ptr(), C.byref(self._shape(B)), C.byref(tg),
                                                      grad_loss.data_ptr(), grad_head.data_ptr(), self._stream()),
                           "ppn_loss_backward")
            else:
                _lib.check(self.lib.ppn_loss_backward_opt(feature_map.data_ptr(), C.byref(self._shape(B, opt[0])), C.byref(tg),
                                                          C.byref(opt[1]), grad_loss.data_ptr(), grad_head.data_ptr(),
                                                          self._stream()),
                           "ppn_loss_backward_opt")
        return grad_head
