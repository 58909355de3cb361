"""Host side of the B200 pose parser: torch tensors in, packed humans out.

:class:`PoseParser` owns the device buffers (torch is used for memory and streams only) and
calls the C ABI in ``libppn_decode.so`` through ctypes.  The batched entry
:meth:`PoseParser.parse` takes the un-sliced head tensor ``out[B, C, H, W]`` straight from
``PoseProposalNet.forward`` (model.py:104-136) so the seven ``.cpu().numpy()`` copies of
rt_test.py:109-120 disappear; :class:`PackedHumans` converts the packed result back into the
reference's ``(humans, scores)`` lists of dicts (datatest.py:98-132) on request.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from typing import List, Optional, Tuple

import numpy as np
import torch

from . import _lib
from .config import PPNConfig


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream_ptr(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class _CConfig:
    """ctypes views of a PPNConfig; keeps the chain arrays alive."""

    def __init__(self, cfg: PPNConfig, n_nms_parts: int = 1):
        self.cfg = cfg
        self.off, self.limb, self.part = cfg.chains()
        if len(self.off) - 1 > _lib.MAX_CHAINS or len(self.limb) > _lib.MAX_CHAIN_STEPS:
            raise ValueError("too many / too long track orders for the kernel argument table")
        gW, gH = cfg.gridsize
        self._shape_fields = dict(K=cfg.K, E=cfg.E, H=cfg.H, W=cfg.W, sH=cfg.sH, sW=cfg.sW, inW=cfg.inW, inH=cfg.inH,
                                  gridW=gW, gridH=gH, off_h=cfg.off_h, off_w=cfg.off_w)
        self.n_nms_parts = int(n_nms_parts)
        self._params = {}             # flag mask -> PPNParams
        self.params = self.params_for(0)

    def params_for(self, flags: int) -> _lib.PPNParams:
        """The PPNParams carrying the PPN_FLAG_* mask `flags` (built once per mask, then reused)."""
        p = self._params.get(int(flags))
        if p is None:
            p = self._params[int(flags)] = self._make_params(self.cfg, self.n_nms_parts, int(flags))
        return p

    @staticmethod
    def flags(input_complete: bool = False, clear_unused: bool = False) -> int:
        return (_lib.FLAG_INPUT_COMPLETE if input_complete else 0) | (_lib.FLAG_CLEAR_UNUSED if clear_unused else 0)

    def _make_params(self, cfg, n_nms_parts, flags):
        # numpy demotes the Python-float thresholds to fp32 when comparing with fp32 arrays
        return _lib.PPNParams(
            float(np.float32(cfg.detection_thresh)), float(np.float32(cfg.nms_thresh)), int(cfg.min_num_keypoints),
            int(n_nms_parts), len(self.off) - 1, int(flags),
            self.off.ctypes.data_as(_lib.i32p), self.limb.ctypes.data_as(_lib.i32p), self.part.ctypes.data_as(_lib.i32p))

    def shape(self, B: int, head_dtype: int = 0) -> _lib.PPNShape:
        return _lib.PPNShape(B=B, head_dtype=head_dtype, **self._shape_fields)


class PackedHumans:
    """Fixed-stride packed result (layout of ``PPNHumans`` in include/ppn_decode.h).

    ``count[b]`` humans of image ``b`` sit in slots ``[0, count[b])`` in the reference's list
    order (descending root score).  Tensors stay where the parser wrote them (device for
    :meth:`PoseParser.parse`, host for :meth:`PoseParser.parse_host`) until asked.
    """

    def __init__(self, cfg: PPNConfig, count, root_cell, part_cell, part_score, part_box):
        self.cfg = cfg
        self.count, self.root_cell, self.part_cell = count, root_cell, part_cell
        self.part_score, self.part_box = part_score, part_box

    @property
    def R(self) -> int:
        return self.root_cell.shape[1]

    def cpu(self) -> "PackedHumans":
        if self.count.device.type == "cpu":
            return self
        return PackedHumans(self.cfg, *(t.cpu() for t in (self.count, self.root_cell, self.part_cell,
                                                           self.part_score, self.part_box)))

    def numpy(self):
        h = self.cpu()
        return {k: getattr(h, k).numpy() for k in ("count", "root_cell", "part_cell", "part_score", "part_box")}

    def numpy_used(self):
        """Like :meth:`numpy`, but only the slots that carry humans cross to the host: the counts first, then the
        first max(count) slots of every array (what :meth:`to_lists` needs; the rest of the R slots is padding)."""
        count = self.count.cpu().numpy()
        m = int(min(int(count.max()) if count.size else 0, self.R))
        take = lambda t: (t if t.device.type == "cpu" else t[:, :m].cpu()).numpy()
        return {"count": count, "root_cell": take(self.root_cell), "part_cell": take(self.part_cell),
                "part_score": take(self.part_score), "part_box": take(self.part_box)}

    def humans(self, b: int = 0):
        """(humans, scores) of image ``b`` exactly as ``get_humans_by_feature`` returns them:
        dicts keyed by part id in first-insertion order, fp32 ``(ymin,xmin,ymax,xmax)`` boxes."""
        return self.to_lists()[b]

    def to_lists(self) -> List[Tuple[list, list]]:
        a = self.numpy_used()
        graphs = self.cfg.directed_graphs
        K = self.cfg.K
        result = []
        for b in range(a["count"].shape[0]):
            n = int(a["count"][b])
            if n > self.R:
                raise RuntimeError(f"image {b}: {n} humans but only {self.R} slots were provided")
            humans, scores = [], []
            for i in range(n):
                cell = a["part_cell"][b, i]
                keys = [0]
                for _, ts in graphs:                       # insertion order of datatest.py:104-125
                    for t in ts:
                        if cell[t] < 0:
                            break
                        if t not in keys:
                            keys.append(t)
                assert len(keys) == int((cell[:K] >= 0).sum()), "track orders do not form a tree"
                humans.append({t: a["part_box"][b, i, t].copy() for t in keys})
                scores.append({t: np.float32(a["part_score"][b, i, t]) for t in keys})
            result.append((humans, scores))
        return result


def unpack_entries(buf, B: int, cap_entries: int, offsets, derive: bool = False):
    """Host view of one dense entry buffer (see include/ppn_decode.h, ppn_pack_humans).

    buf: uint8 numpy array or CPU tensor.  Returns dict(total, overflow, count[B] humans per image,
    entries[B] per image, start[B] first entry of each image, part[cap], cell[cap], score[cap],
    box[cap,4]).  Within an image an entry with part 0 starts a new human."""
    a = buf.numpy() if isinstance(buf, torch.Tensor) else np.asarray(buf)
    o_h, o_i, o_s, o_b = offsets
    header = a[o_h:o_h + 4 * (2 + 3 * B)].view(np.int32)
    count, entries, start = header[2:2 + B], header[2 + B:2 + 2 * B], header[2 + 2 * B:2 + 3 * B].astype(np.int64)
    idcell = a[o_i:o_i + 4 * cap_entries].view(np.uint32)
    score = a[o_s:o_s + 4 * cap_entries].view(np.float32)
    box = a[o_b:o_b + 16 * cap_entries].view(np.float32).reshape(cap_entries, 4)
    if derive:          # a buffer written remotely (ppn_parse_dense_remote) carries the table but not header[0..1]
        total, overflow = int(entries.sum()), bool(((start + entries) > cap_entries).any())
    else:
        total, overflow = int(header[0]), bool(header[1])
    return dict(total=total, overflow=overflow, count=count, entries=entries, start=start,
                part=(idcell >> 16).astype(np.int32), cell=(idcell & 0xffff).astype(np.int32), score=score, box=box)


def entries_to_packed(rec, b: int, K: int):
    """Rebuild image b's fixed-K arrays (part_cell [n,K], part_score [n,K], part_box [n,K,4]) from
    unpack_entries() output — the inverse of the packing, for consumers and tests."""
    s0, n_e = int(rec["start"][b]), int(rec["entries"][b])
    part, cell = rec["part"][s0:s0 + n_e], rec["cell"][s0:s0 + n_e]
    human = np.cumsum(part == 0) - 1                       # entry -> human index within the image
    n = int(human[-1]) + 1 if n_e else 0
    pc = np.full((n, K), -1, np.int32)
    ps = np.zeros((n, K), np.float32)
    pb = np.zeros((n, K, 4), np.float32)
    pc[human, part] = cell
    ps[human, part] = rec["score"][s0:s0 + n_e]
    pb[human, part] = rec["box"][s0:s0 + n_e]
    return pc, ps, pb


class CapturedParse:
    """A recorded ``PoseParser.parse`` (see :meth:`PoseParser.capture`): ``replay()`` re-runs it on the captured
    ``head`` / ``out`` buffers."""

    def __init__(self, graph, head: torch.Tensor, out: PackedHumans):
        self.graph, self.head, self.out = graph, head, out

    def replay(self) -> PackedHumans:
        self.graph.replay()
        return self.out


class PoseParser:
    """Decode + NMS + limb arg-max + tree parse of PPN head tensors on one B200.

    Not thread-safe per instance (buffers are reused); make one per stream/thread.
    """

    def __init__(self, cfg: PPNConfig, device=None, max_humans: Optional[int] = None, n_nms_parts: int = 1):
        if cfg.HW > _lib.MAX_CELLS:
            raise ValueError(f"grid of {cfg.HW} cells exceeds the kernels' limit of {_lib.MAX_CELLS}")
        self.cfg = cfg
        self.lib = _lib.lib()                      # raises if the CUDA library is missing
        if not torch.cuda.is_available():
            raise RuntimeError("PoseParser needs a CUDA device; there is no CPU path")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.R = int(max_humans) if max_humans else cfg.HW
        self.n_nms_parts = int(n_nms_parts)
        self.c = _CConfig(cfg, self.n_nms_parts)
        self._ws = None
        self._ws_need = {}            # B -> workspace bytes (ppn_workspace_bytes is pure arithmetic)
        self._shapes = {}             # B -> PPNShape
        self._layouts = {}            # (B, cap) -> dense record layout
        self._out = None
        self._out_B = 0
        self._host_scratch = None

    def _guard(self):
        """Make the parser's device current for the C call (no-op when it already is)."""
        if torch.cuda.current_device() == self.device.index:
            return contextlib.nullcontext()
        return torch.cuda.device(self.device)

    def _shape(self, B: int, dtype: int = 0) -> _lib.PPNShape:
        s = self._shapes.get((B, dtype))
        if s is None:
            s = self._shapes[(B, dtype)] = self.c.shape(B, dtype)
        return s

    # ---- buffers --------------------------------------------------------------------- #
    _DTYPES = {torch.float32: _lib.HEAD_F32, torch.float16: _lib.HEAD_F16, torch.bfloat16: _lib.HEAD_BF16}

    def _check_head(self, head: torch.Tensor) -> int:
        cfg = self.cfg
        if head.dtype not in self._DTYPES or head.dim() != 4 or tuple(head.shape[1:]) != (cfg.C, cfg.H, cfg.W):
            raise ValueError(f"head must be fp32/fp16/bf16 [B,{cfg.C},{cfg.H},{cfg.W}], got {head.dtype} {tuple(head.shape)}")
        if not head.is_contiguous():
            raise ValueError("head must be contiguous NCHW")
        return head.shape[0]

    def _workspace(self, B: int) -> torch.Tensor:
        need = self._ws_need.get(B)
        if need is None:
            n = C.c_size_t()
            _lib.check(self.lib.ppn_workspace_bytes(C.byref(self._shape(B)), C.byref(self.c.params), C.byref(n)),
                       "ppn_workspace_bytes")
            need = self._ws_need[B] = n.value
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 256), dtype=torch.uint8, device=self.device)
        return self._ws

    def alloc_output(self, B: int, device=None, pin: bool = False) -> PackedHumans:
        dev = self.device if device is None else torch.device(device)
        kw = dict(device=dev, pin_memory=pin) if dev.type == "cpu" else dict(device=dev)
        K, R = self.cfg.K, self.R
        return PackedHumans(self.cfg,
                            torch.zeros(B, dtype=torch.int32, **kw),
                            torch.empty(B, R, dtype=torch.int32, **kw),
                            torch.empty(B, R, K, dtype=torch.int32, **kw),
                            torch.empty(B, R, K, dtype=torch.float32, **kw),
                            torch.empty(B, R, K, 4, dtype=torch.float32, **kw))

    def _humans_struct(self, out: PackedHumans) -> _lib.PPNHumans:
        return _lib.PPNHumans(out.count.data_ptr(), out.root_cell.data_ptr(), out.part_cell.data_ptr(),
                              out.part_score.data_ptr(), out.part_box.data_ptr(), out.R)

    # ---- the whole path ---------------------------------------------------------------- #
    def parse(self, head: torch.Tensor, out: Optional[PackedHumans] = None, input_complete: bool = False,
              dense: Optional[torch.Tensor] = None, cap_entries: int = 0, skip_slots: bool = False,
              remote: Optional[Tuple[int, int]] = None, clear_unused: bool = False) -> PackedHumans:
        """Enqueue the whole path for a device batch on torch's current stream (asynchronous).

        ``out`` may be a preallocated :meth:`alloc_output` to reuse; otherwise the parser's own
        buffer is returned and overwritten by the next call.

        ``input_complete=True`` (``PPN_FLAG_INPUT_COMPLETE``) is a promise that ``head`` was fully
        written before this call — e.g. it has been resident since an earlier, finished step — not
        just ordered before it on the stream by a producer kernel that may still be running.  The
        call may then overlap the previous ``parse`` on this stream (its arg-max streams while the
        previous call's tree parse finishes); give consecutive overlapping calls different ``out``.

        ``dense`` (a uint8 device buffer of ``packed_layout(B, cap_entries)`` bytes): also produce the
        dense (human, part) entry buffer of the multi-GPU gather (``ppn_parse_dense``); with
        ``skip_slots`` the fixed-stride arrays of ``out`` other than ``count`` may be left unwritten.

        ``remote = (address, bytes)`` of ANOTHER dense buffer of the same layout — e.g. the gather root's,
        peer-mapped over NVLink (:class:`..sharded.PeerPoseGatherer`): the parse kernel stores the per-image
        table and the entries there (``ppn_parse_dense_remote``); ``dense`` then only needs to hold the header.

        ``clear_unused`` (``PPN_FLAG_CLEAR_UNUSED``): slots past ``count[b]`` are reset (-1 / 0) instead of keeping
        whatever ``out`` held.  It combines with ``input_complete``.
        """
        B = self._check_head(head)
        if head.device != self.device:
            raise ValueError(f"head is on {head.device}, parser on {self.device}")
        if out is None:
            if self._out is None or self._out_B < B:
                self._out, self._out_B = self.alloc_output(B), B
            o = self._out
            out = o if self._out_B == B else PackedHumans(self.cfg, o.count[:B], o.root_cell[:B], o.part_cell[:B],
                                                          o.part_score[:B], o.part_box[:B])
        ws = self._workspace(B)
        hs = self._humans_struct(out)
        with self._guard():
            params = self.c.params_for(_CConfig.flags(input_complete, clear_unused))
            st = torch.cuda.current_stream(self.device).cuda_stream
            if dense is None:
                rc = self.lib.ppn_parse(head.data_ptr(), C.byref(self._shape(B, self._DTYPES[head.dtype])), C.byref(params), C.byref(hs),
                                        ws.data_ptr(), ws.numel(), st)
            elif remote is not None:
                rc = self.lib.ppn_parse_dense_remote(head.data_ptr(), C.byref(self._shape(B, self._DTYPES[head.dtype])), C.byref(params),
                                                     C.byref(hs), dense.data_ptr(), dense.numel(), int(remote[0]), int(remote[1]),
                                                     int(cap_entries), int(bool(skip_slots)), ws.data_ptr(), ws.numel(), st)
            else:
                rc = self.lib.ppn_parse_dense(head.data_ptr(), C.byref(self._shape(B, self._DTYPES[head.dtype])), C.byref(params),
                                              C.byref(hs), dense.data_ptr(), dense.numel(), int(cap_entries), int(bool(skip_slots)),
                                              ws.data_ptr(), ws.numel(), st)
        if rc:
            raise _lib.PPNError(rc, "ppn_parse" if dense is None else ("ppn_parse_dense" if remote is None else "ppn_parse_dense_remote"))
        return out

    def parse_proposals(self, head: torch.Tensor, out: Optional[PackedHumans] = None,
                        clear_unused: bool = False) -> PackedHumans:
        """The proposal-pair parse of a device batch (``ppn_parse_proposals``; asynchronous, on torch's current stream).

        Unlike :meth:`parse`, which walks the arg-max of every limb window from each root as the reference does, this
        parser gives every part NMS-filtered proposals, scores each candidate pair of a limb as
        ``(delta_s * limb) * delta_t`` and matches them greedily down the skeleton tree, so no part instance belongs
        to two humans (DESIGN.md §13).  The result has the layout of :meth:`parse`'s and feeds the same consumers
        (``to_lists``, ``part_centres``, ``skeleton``, ``evaluation.APEvaluator``).  The track orders must form a tree
        rooted at part 0.  ``out`` and ``clear_unused`` as for :meth:`parse`."""
        B = self._check_head(head)
        if head.device != self.device:
            raise ValueError(f"head is on {head.device}, parser on {self.device}")
        if out is None:
            out = self.alloc_output(B)
        shape = self._shape(B, self._DTYPES[head.dtype])
        params = self.c.params_for(_CConfig.flags(clear_unused=clear_unused))
        need = C.c_size_t()
        _lib.check(self.lib.ppn_parse_proposals_workspace_bytes(C.byref(shape), C.byref(params), C.byref(need)),
                   "ppn_parse_proposals_workspace_bytes")
        if getattr(self, "_prop_ws", None) is None or self._prop_ws.numel() < need.value:
            self._prop_ws = torch.empty(max(need.value, 256), dtype=torch.uint8, device=self.device)
        hs = self._humans_struct(out)
        with self._guard():
            _lib.check(self.lib.ppn_parse_proposals(head.data_ptr(), C.byref(shape), C.byref(params), C.byref(hs),
                                                    self._prop_ws.data_ptr(), self._prop_ws.numel(),
                                                    torch.cuda.current_stream(self.device).cuda_stream), "ppn_parse_proposals")
        return out

    def capture(self, head: torch.Tensor, out: Optional[PackedHumans] = None, **parse_kwargs) -> "CapturedParse":
        """Record ``parse(head, out)`` into a CUDA graph for repeated use on the SAME buffers — the single-image
        loop of rt_test.py:87-147, where the network writes its output into one tensor frame after frame: a replay
        is one graph launch instead of two or three kernel launches from Python.  ``head`` (and ``out``) must stay
        alive and in place; refill ``head`` and call ``replay()`` (asynchronous, on torch's current stream)."""
        B = self._check_head(head)
        if out is None:
            out = self.alloc_output(B)
        self.parse(head, out=out, **parse_kwargs)                    # warm-up outside the capture: workspace, attributes
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.graph(graph, stream=side):
            self.parse(head, out=out, **parse_kwargs)
        torch.cuda.current_stream(self.device).wait_stream(side)
        return CapturedParse(graph, head, out)

    def launches_per_parse(self, B: int) -> int:
        shape = self.c.shape(B)
        return int(self.lib.ppn_parse_launches(C.byref(shape), C.byref(self.c.params)))

    def parse_plan(self, B: int) -> dict:
        """How ``parse`` runs a batch of B: launches, sub-batches, the arg-max ring's shared-memory cap, staging."""
        info = (C.c_int32 * 4)()
        _lib.check(self.lib.ppn_parse_plan(C.byref(self.c.shape(B)), C.byref(self.c.params), info), "ppn_parse_plan")
        return dict(launches=info[0], sub_batches=info[1], ring_cap=info[2], staged=bool(info[3]))

    def limb_stream_probe(self, head: torch.Tensor, smem_cap: int = 0) -> None:
        """Run the arg-max kernel's bulk-copy ring over `head` without compares or stores (``ppn_limb_stream_probe``):
        the read ceiling of that access pattern; asynchronous, on torch's current stream."""
        B = self._check_head(head)
        cfg = self.cfg
        if getattr(self, "_probe_amax", None) is None or self._probe_amax.shape[0] < B:
            self._probe_amax = torch.empty(B, cfg.E, cfg.H, cfg.W, dtype=torch.uint16, device=self.device)
        with self._guard():
            _lib.check(self.lib.ppn_limb_stream_probe(head.data_ptr(), C.byref(self._shape(B, self._DTYPES[head.dtype])),
                                                      self._probe_amax.data_ptr(), int(smem_cap),
                                                      torch.cuda.current_stream(self.device).cuda_stream), "ppn_limb_stream_probe")

    def parse_host(self, head: torch.Tensor, out: Optional[PackedHumans] = None, clear_unused: bool = False) -> PackedHumans:
        """The whole path from HOST memory (pinned for full copy speed) to host results;
        synchronous.  This is the end-to-end call with the host<->device copies inside.

        Only the first ``max(count)`` slots of every image are copied back; the others keep what ``out`` held unless
        ``clear_unused`` (``PPN_FLAG_CLEAR_UNUSED``) resets every slot past ``count[b]`` to -1 / 0."""
        B = self._check_head(head)
        if head.device.type != "cpu":
            raise ValueError("parse_host takes a CPU tensor")
        if out is None:
            out = self.alloc_output(B, device="cpu", pin=True)
        need = C.c_size_t()
        shape = self.c.shape(B, self._DTYPES[head.dtype])
        _lib.check(self.lib.ppn_parse_host_scratch_bytes(C.byref(shape), C.byref(self.c.params), self.R, C.byref(need)),
                   "ppn_parse_host_scratch_bytes")
        if self._host_scratch is None or self._host_scratch.numel() < need.value:
            self._host_scratch = torch.empty(need.value, dtype=torch.uint8, device=self.device)
        hs = self._humans_struct(out)
        params = self.c.params_for(_CConfig.flags(clear_unused=clear_unused))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ppn_parse_host(_ptr(head), C.byref(shape), C.byref(params), C.byref(hs),
                                               _ptr(self._host_scratch), self._host_scratch.numel()), "ppn_parse_host")
        return out

    # ---- the network head fused in: conv3 (1x1) + sigmoid + parse (model.py:85, 133-136) ------------ #
    _OPERANDS = {"tf32": _lib.GEMM_TF32, "f16": _lib.GEMM_F16, "bf16": _lib.GEMM_BF16}

    def _check_features(self, feat, weight, bias, operand="tf32"):
        """-> (B, Cin, PPNHeadOptions).  feat: fp32 NCHW contiguous, or — 16-bit operands only — a 16-bit tensor of
        the operand type whose memory is [B, H, W, Cin] (torch.channels_last), read in place."""
        cfg = self.cfg
        if operand not in self._OPERANDS:
            raise ValueError(f"operand must be one of {sorted(self._OPERANDS)}, got {operand!r}")
        if feat.dim() != 4 or tuple(feat.shape[2:]) != (cfg.H, cfg.W):
            raise ValueError(f"feat must be [B, Cin, {cfg.H}, {cfg.W}], got {tuple(feat.shape)}")
        want16 = {"f16": torch.float16, "bf16": torch.bfloat16}.get(operand)
        if feat.dtype == torch.float32 and feat.is_contiguous():
            layout = _lib.FEAT_NCHW_F32
        elif want16 is not None and feat.dtype == want16 and feat.permute(0, 2, 3, 1).is_contiguous():
            layout = _lib.FEAT_NHWC_16
        else:
            raise ValueError("feat must be contiguous fp32 NCHW" + (f" or channels_last {want16}" if want16 else "") +
                             f", got {feat.dtype} with strides {feat.stride()}")
        Cin = feat.shape[1]
        w2 = weight.reshape(weight.shape[0], -1)
        if weight.dtype != torch.float32 or tuple(w2.shape) != (cfg.C, Cin) or not w2.is_contiguous():
            raise ValueError(f"weight must be contiguous fp32 [{cfg.C}, {Cin}(, 1, 1)], got {weight.dtype} {tuple(weight.shape)}")
        if bias is not None and (bias.dtype != torch.float32 or tuple(bias.shape) != (cfg.C,) or not bias.is_contiguous()):
            raise ValueError(f"bias must be contiguous fp32 [{cfg.C}]")
        for t in (feat, weight, bias):
            if t is not None and t.device != self.device:
                raise ValueError(f"tensor on {t.device}, parser on {self.device}")
        return feat.shape[0], Cin, _lib.PPNHeadOptions(self._OPERANDS[operand], layout)

    def _emit_buffers(self, B: int, emit: bool):
        if not emit:
            return None, None
        cfg = self.cfg
        return (torch.empty(B, cfg.C, cfg.H, cfg.W, dtype=torch.float32, device=self.device),
                torch.empty(B, cfg.C, cfg.H, cfg.W, dtype=torch.float32, device=self.device))

    def _head_workspace(self, B: int, Cin: int, opt) -> torch.Tensor:
        need = C.c_size_t()
        _lib.check(self.lib.ppn_head_workspace_bytes_opt(C.byref(self._shape(B)), Cin, C.byref(opt), C.byref(need)),
                   "ppn_head_workspace_bytes_opt")
        if getattr(self, "_head_ws", None) is None or self._head_ws.numel() < need.value:
            self._head_ws = torch.empty(max(need.value, 256), dtype=torch.uint8, device=self.device)
        return self._head_ws

    def head_gemm_argmax(self, feat: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, emit: bool = False,
                         operand: str = "tf32"):
        """The fused head kernel alone (``ppn_head_gemm_argmax_opt``): 1x1 convolution on the tensor cores, sigmoid and
        limb-window arg-max in the epilogue.  -> (dec [B, 6K, H, W] fp32, amax [B, E, H, W] uint16, logits, head);
        the last two are the convolution output and its sigmoid [B, C, H, W] when ``emit`` (parity tests), else None.
        ``operand``: "tf32" (fp32 activations read in place), "f16" or "bf16" (see ``parse_features``)."""
        B, Cin, opt = self._check_features(feat, weight, bias, operand)
        cfg = self.cfg
        dec = torch.empty(B, 6 * cfg.K, cfg.H, cfg.W, dtype=torch.float32, device=self.device)
        amax = torch.empty(B, cfg.E, cfg.H, cfg.W, dtype=torch.uint16, device=self.device)
        logits, head = self._emit_buffers(B, emit)
        ws = self._head_workspace(B, Cin, opt)
        with self._guard():
            _lib.check(self.lib.ppn_head_gemm_argmax_opt(feat.data_ptr(), weight.data_ptr(), _ptr(bias), Cin, C.byref(self._shape(B)),
                                                         C.byref(opt), ws.data_ptr(), ws.numel(), dec.data_ptr(), amax.data_ptr(),
                                                         _ptr(logits), _ptr(head), torch.cuda.current_stream(self.device).cuda_stream),
                       "ppn_head_gemm_argmax_opt")
        return dec, amax, logits, head

    def parse_features(self, feat: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
                       out: Optional[PackedHumans] = None, emit: bool = False, operand: str = "tf32",
                       clear_unused: bool = False):
        """``sigmoid(conv3(feat))`` parsed into humans without the head tensor ever being written
        (``ppn_head_parse_opt``): feat = the input of the network's last layer [B, Cin, H, W] (model.py:133), weight /
        bias = ``conv3``'s.  ``operand`` picks the tensor-core operand type: "tf32" (default: fp32 activations read in
        place, the precision of the reference's conv under PyTorch's defaults), "f16" or "bf16" (operands rounded to 16
        bits, fp32 accumulation — the reference's conv under its AMP setup, main.py:282-289; feat may then also be a
        channels_last tensor of that type, read in place).  Asynchronous on torch's current stream.
        -> PackedHumans, or (PackedHumans, logits, head) when ``emit`` — the kernel then also writes the convolution
        output and its sigmoid for parity checks.  ``clear_unused``: as for :meth:`parse`."""
        B, Cin, opt = self._check_features(feat, weight, bias, operand)
        if out is None:
            out = self.alloc_output(B)
        ws = self._head_workspace(B, Cin, opt)
        logits, head = self._emit_buffers(B, emit)
        hs = self._humans_struct(out)
        params = self.c.params_for(_CConfig.flags(clear_unused=clear_unused))
        with self._guard():
            _lib.check(self.lib.ppn_head_parse_opt(feat.data_ptr(), weight.data_ptr(), _ptr(bias), Cin, C.byref(self._shape(B)),
                                                   C.byref(params), C.byref(opt), C.byref(hs), ws.data_ptr(), ws.numel(),
                                                   _ptr(logits), _ptr(head), torch.cuda.current_stream(self.device).cuda_stream),
                       "ppn_head_parse_opt")
        return (out, logits, head) if emit else out

    def capture_features(self, feat: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
                         out: Optional[PackedHumans] = None, operand: str = "tf32") -> "CapturedParse":
        """Record ``parse_features(feat, weight, bias, out)`` into a CUDA graph for repeated use on the SAME buffers
        (the single-image loop of rt_test.py:87-147 with the backbone writing ``feat`` in place): a replay is one graph
        launch instead of four or five launches from Python.  All tensors must stay alive and in place."""
        B, _, _ = self._check_features(feat, weight, bias, operand)
        if out is None:
            out = self.alloc_output(B)
        self.parse_features(feat, weight, bias, out=out, operand=operand)      # warm-up outside the capture: workspace, attributes
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.graph(graph, stream=side):
            self.parse_features(feat, weight, bias, out=out, operand=operand)
        torch.cuda.current_stream(self.device).wait_stream(side)
        cap = CapturedParse(graph, feat, out)
        cap.keep = (weight, bias, self._head_ws)                               # the graph holds their addresses
        return cap

    # ---- keypoints (what drawing and AP evaluation read off the boxes) ------------------- #
    def part_centres(self, humans: PackedHumans) -> torch.Tensor:
        """fp32 [B, R, K, 2] = (y, x) centre of every part's box, (0, 0) where absent
        (datatest.py:200-211, 314-317); asynchronous, on torch's current stream."""
        B = humans.count.shape[0]
        out = torch.empty(B, humans.R, self.cfg.K, 2, dtype=torch.float32, device=self.device)
        hs = self._humans_struct(humans)
        with self._guard():
            _lib.check(self.lib.ppn_part_centres(C.byref(hs), B, self.cfg.K, out.data_ptr(),
                                                 torch.cuda.current_stream(self.device).cuda_stream), "ppn_part_centres")
        return out

    def skeleton(self, humans: PackedHumans, edges=None):
        """Drawing primitives of every slot (``ppn_skeleton``; datatest.py:162-232): -> (rect [B, R, 4] int32
        (xmin, ymin, xmax, ymax), keypoint [B, R, K, 2] fp32 (x, y), segment [B, R, E, 4] fp32 (bx, by, ex, ey));
        NaN where a part / limb is absent.  Asynchronous, on torch's current stream."""
        cfg = self.cfg
        if edges is None:
            from . import config as pcfg
            edges = {(18, 17): pcfg.EDGES, (16, 15): pcfg.EDGES_16}.get((cfg.K, cfg.E))
            if edges is None:
                raise ValueError("pass `edges` ([E][2] part ids) for a skeleton that is not one of config.py's")
        e = np.ascontiguousarray(np.asarray(edges, np.int32).reshape(-1, 2))
        if e.shape[0] != cfg.E:
            raise ValueError(f"{e.shape[0]} edges for a configuration with E = {cfg.E}")
        B = humans.count.shape[0]
        rect = torch.empty(B, humans.R, 4, dtype=torch.int32, device=self.device)
        kp = torch.empty(B, humans.R, cfg.K, 2, dtype=torch.float32, device=self.device)
        seg = torch.empty(B, humans.R, cfg.E, 4, dtype=torch.float32, device=self.device)
        hs = self._humans_struct(humans)
        with self._guard():
            _lib.check(self.lib.ppn_skeleton(C.byref(hs), B, cfg.K, cfg.E, e.ctypes.data_as(_lib.i32p), rect.data_ptr(),
                                             kp.data_ptr(), seg.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream),
                       "ppn_skeleton")
        return rect, kp, seg

    # ---- dense entries (what the multi-GPU gather ships) -------------------------------- #
    def packed_layout(self, B: int, cap_entries: int):
        """-> (bytes, (header, idcell, score, box) byte offsets) of the dense entry buffer."""
        key = (B, cap_entries)
        hit = self._layouts.get(key)
        if hit is not None:
            return hit
        nbytes = C.c_size_t()
        offs = (C.c_size_t * 4)()
        _lib.check(self.lib.ppn_packed_bytes(B, cap_entries, C.byref(nbytes), offs), "ppn_packed_bytes")
        self._layouts[key] = (nbytes.value, tuple(int(o) for o in offs))
        return self._layouts[key]

    def pack(self, humans: PackedHumans, cap_entries: int, buf: Optional[torch.Tensor] = None,
             stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """Compact the fixed-stride result into one contiguous uint8 buffer (asynchronous): counts
        plus one dense (part, cell, score, box) entry per PRESENT part, `cap_entries` at most
        (ppn_pack_humans).  Runs on `stream` (default: torch's current stream)."""
        B = humans.count.shape[0]
        nbytes, _ = self.packed_layout(B, cap_entries)
        if buf is None:
            buf = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        hs = self._humans_struct(humans)
        with self._guard():
            st = (stream if stream is not None else torch.cuda.current_stream(self.device)).cuda_stream
            _lib.check(self.lib.ppn_pack_humans(C.byref(hs), B, self.cfg.K, cap_entries, buf.data_ptr(), buf.numel(), st),
                       "ppn_pack_humans")
        return buf

    # ---- single stages (what the stage-level parity tests call) ------------------------- #
    def limb_argmax(self, head: torch.Tensor) -> torch.Tensor:
        """uint16 [B, E, H, W]: first arg-max of every limb window (datatest.py:100,113)."""
        B = self._check_head(head)
        cfg = self.cfg
        amax = torch.empty(B, cfg.E, cfg.H, cfg.W, dtype=torch.uint16, device=self.device)
        shape = self.c.shape(B, self._DTYPES[head.dtype])
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ppn_limb_argmax(_ptr(head), C.byref(shape), _ptr(amax), _stream_ptr(self.device)), "ppn_limb_argmax")
        return amax

    def limb_argmax_into(self, head: torch.Tensor, amax: Optional[torch.Tensor] = None) -> torch.Tensor:
        """:meth:`limb_argmax` into a caller's (or a cached) buffer: nothing is allocated per call (benchmarks)."""
        B = self._check_head(head)
        cfg = self.cfg
        if amax is None:
            if getattr(self, "_probe_amax", None) is None or self._probe_amax.shape[0] < B:
                self._probe_amax = torch.empty(B, cfg.E, cfg.H, cfg.W, dtype=torch.uint16, device=self.device)
            amax = self._probe_amax
        with self._guard():
            _lib.check(self.lib.ppn_limb_argmax(head.data_ptr(), C.byref(self._shape(B, self._DTYPES[head.dtype])), amax.data_ptr(),
                                                torch.cuda.current_stream(self.device).cuda_stream), "ppn_limb_argmax")
        return amax

    def decode_candidates(self, head: torch.Tensor, n_parts: int = 1, detection_thresh: Optional[float] = None):
        """-> (cell [B,P,HW] i32, score [B,P,HW] f32, box [B,P,HW,4] f32, count [B,P] i32)."""
        B = self._check_head(head)
        HW = self.cfg.HW
        thr = float(np.float32(self.cfg.detection_thresh if detection_thresh is None else detection_thresh))
        cell = torch.empty(B, n_parts, HW, dtype=torch.int32, device=self.device)
        score = torch.empty(B, n_parts, HW, dtype=torch.float32, device=self.device)
        box = torch.empty(B, n_parts, HW, 4, dtype=torch.float32, device=self.device)
        count = torch.empty(B, n_parts, dtype=torch.int32, device=self.device)
        shape = self.c.shape(B, self._DTYPES[head.dtype])
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ppn_decode_candidates(_ptr(head), C.byref(shape), n_parts, thr, _ptr(cell), _ptr(score),
                                                      _ptr(box), _ptr(count), _stream_ptr(self.device)), "ppn_decode_candidates")
        return cell, score, box, count

    def nms(self, box: torch.Tensor, score: Optional[torch.Tensor], count: torch.Tensor, thresh: float,
            limit: Optional[int] = None):
        """box [P, stride, 4], score [P, stride] or None, count [P] -> (keep_idx [P, stride], keep_count [P])."""
        n_prob, stride = box.shape[0], box.shape[1]
        keep = torch.empty(n_prob, stride, dtype=torch.int32, device=self.device)
        kcount = torch.empty(n_prob, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ppn_nms(_ptr(box), _ptr(score), _ptr(count), n_prob, stride, float(np.float32(thresh)),
                                        int(limit or 0), _ptr(keep), _ptr(kcount), _stream_ptr(self.device)), "ppn_nms")
        return keep, kcount

    def tree_parse(self, head, amax, cand_cell, keep_idx, keep_count, out: Optional[PackedHumans] = None) -> PackedHumans:
        B = self._check_head(head)
        if out is None:
            out = self.alloc_output(B)
        shape, hs = self.c.shape(B, self._DTYPES[head.dtype]), self._humans_struct(out)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ppn_tree_parse(_ptr(head), C.byref(shape), C.byref(self.c.params), _ptr(amax), _ptr(cand_cell),
                                               _ptr(keep_idx), _ptr(keep_count), C.byref(hs), _stream_ptr(self.device)), "ppn_tree_parse")
        return out
