"""Drop-in host side of the reference's `model.py` for the GGNN role-graph stage.

`FCGGNN(encoder, D_hidden_state)` keeps the reference's constructor, attribute / parameter names (= checkpoint
keys), `forward(img, gt_verb)`, `predict_verb`, `predict_nouns`, `verb_loss`, `nouns_loss` (model.py:90-201) and
`GGSNN(layersize).forward(hidden_state, mask, verb)` (model.py:38-86), each differentiable on its own: in bf16 mode a
caller can train through `model.ggsnn(node, mask)` with its own node init, adjacency or losses, and the fused paths
return dL/dfeatures, so an unfrozen backbone (`model.convnet_nouns.requires_grad_(True)`), a trainable adapter in front
of `forward_features` or a saliency map dL/dimage get their gradients.  The arithmetic of the
stage runs in libsrggnn.so (hand-written sm_100a kernels) through ctypes; PyTorch only owns memory, streams and autograd
bookkeeping.  There is no CPU / eager fallback: non-CUDA inputs raise.

Differences a caller can observe (all documented in DESIGN.md):
  * logits are returned in fp32 as `[..., :n]` views of buffers padded to a multiple of 256 columns;
  * on CUDA the reference always runs under fp16 autocast; this module computes with bf16 tensor-core operands and
    fp32 accumulation/state (`precision="bf16"`), or a 3-term bf16 split that meets fp32 parity
    (`precision="fp32"`, forward only);
  * `model.module` returns the model itself so that unmodified `sr.py` CUDA branches (`model.module.verb_loss`)
    keep working without `nn.DataParallel`.
"""
import ctypes
import os
import warnings
from collections import namedtuple

import torch
import torch.nn as nn

from . import _lib
from ._lib import SRG_MODE_NOUN, SRG_MODE_VERB, SRG_PREC_BF16, SRG_PREC_FP32
from .imsitu_encoder import tables_from_encoder

T_STEPS = 4  # model.py:60
_POISON_WS = os.environ.get("SRG_POISON_WS", "0") == "1"


Situations = namedtuple("Situations", ["verbs", "verb_logp", "labels", "label_logp", "score"])
Situations.__doc__ = """Top-k situations of a batch (FCGGNN.situations_from_features / predict_situations).
    verbs [B,k] int64 (descending verb logit, ties to the lower id); verb_logp [B,k] fp32 log-softmax over the verbs, or
    None when the verbs were given; labels [B,k,R] int64 top-1 label per role slot, -1 on pad slots; label_logp [B,k,R]
    fp32 its log-softmax over the labels, 0 on pad slots; score [B,k] = verb_logp + sum over the real slots of
    label_logp (label term only when the verbs were given).
    FCGGNN.nbest_situations_from_features returns the same fields for the n best situations of each image, which may
    repeat a verb with other labels: verbs / verb_logp [B,n], labels / label_logp [B,n,R], score [B,n] descending."""

MAX_TOPK = 16
MAX_VERB_BEAM = MAX_TOPK - 1      # the n-best decode also reads the log-prob of the best verb outside the beam


def _pad256(n):
    return (n + 255) // 256 * 256


class resnet(nn.Module):
    """torchvision ResNet-152 returning the 2048-d pooled features (model.py:8-35), frozen as in the reference;
    `requires_grad_(True)` fine-tunes it (the stages return dL/dfeatures).  Stock library module, not part of the CUDA
    path; timed separately.  Offline, the pretrained weights cannot be downloaded, so
    `pretrained=None` tries and falls back to random init with a warning."""

    def __init__(self, out_layers, pretrained=None):
        super().__init__()
        import torchvision as tv
        weights = None
        if pretrained is None or pretrained:
            try:
                self.model = tv.models.resnet152(weights=tv.models.ResNet152_Weights.IMAGENET1K_V1, progress=False)
                weights = "imagenet"
            except Exception as e:  # no network / no cached checkpoint
                if pretrained:
                    raise
                warnings.warn("pretrained ResNet-152 weights unavailable (%s); using random init" % type(e).__name__)
        if weights is None:
            self.model = tv.models.resnet152(weights=None)
        for p in self.model.parameters():
            p.requires_grad = False
        self.model.fc = nn.Identity()

    def forward(self, x):
        return self.model(x)


class _Engine:
    """Owns the libsrggnn handle of one model on one device and keeps the packed bf16 weights in sync."""

    def __init__(self, model, device):
        self.lib = _lib.load()
        enc = model.encoder
        self.D = model.D
        self.R = enc.get_max_role_count()
        self.V, self.NR, self.L = enc.get_num_verbs(), enc.get_num_roles(), enc.get_num_labels()
        self.Vpad, self.Lpad = _pad256(self.V), _pad256(self.L)
        self.device = device
        h = ctypes.c_void_p()
        with torch.cuda.device(device):
            _lib.check(self.lib.srg_create(ctypes.byref(h), device.index if device.index is not None else
                                           torch.cuda.current_device(), self.D, self.R, T_STEPS, self.V, self.NR,
                                           self.L))
        self.h = h
        v2r, rc = tables_from_encoder(enc)
        _lib.check(self.lib.srg_set_tables(self.h, v2r.ctypes.data_as(ctypes.c_void_p),
                                           rc.ctypes.data_as(ctypes.c_void_p)))
        self._packed_key = None
        self.pack_gen = 0          # bumped whenever the packed operands are rebuilt (a backward pass must see the
                                   # operands its forward pass ran with)
        self.launches = 0
        self._deferred = False     # srg_set_deferred_chain state of the handle
        self._pending = None       # direct-gradient backward pass in flight: {"grads", "events"}
        self._events = []

    def __del__(self):
        try:
            if self.h:
                self.lib.srg_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def set_cta_group(self, cg):
        _lib.check(self.lib.srg_set_cta_group(self.h, cg))

    def set_compact_rows(self, on):
        """Role-graph rows: real role nodes + one shared pad row (default) or the reference's R rows per image."""
        _lib.check(self.lib.srg_set_compact_rows(self.h, int(bool(on))))

    def param_list(self, model):
        g = model.ggsnn
        return [g.W_p.weight, g.W_p.bias, g.W_z.weight, g.W_z.bias, g.U_z.weight, g.U_z.bias,
                g.W_r.weight, g.W_r.bias, g.U_r.weight, g.U_r.bias, g.W_h.weight, g.W_h.bias,
                g.U_h.weight, g.U_h.bias,
                model.verb_classifier[1].weight, model.verb_classifier[1].bias,
                model.nouns_classifier[1].weight, model.nouns_classifier[1].bias]

    def ensure_packed(self, model, prec):
        params = self.param_list(model)
        flat = getattr(model, "_flat", None)
        key = (prec, getattr(flat, "version", 0)) + tuple((p.data_ptr(), p._version) for p in params)
        if key == self._packed_key:
            return
        for p in params:
            if p.dtype != torch.float32 or not p.is_contiguous() or p.device != self.device:
                raise _lib.SrgError("GGNN parameters must be contiguous fp32 tensors on %s" % self.device)
        sp = _lib.SrgParams(*[ctypes.c_void_p(p.data_ptr()) for p in params])
        _lib.check(self.lib.srg_pack_weights(self.h, ctypes.byref(sp), prec, self.stream()))
        self._packed_key = key
        self.pack_gen += 1

    def check_pack_gen(self, gen):
        if gen != self.pack_gen:
            raise _lib.SrgError("the packed weights changed between this path's forward and its backward pass (another "
                                "forward after a parameter update, or a different precision): gradients would be "
                                "inconsistent -- run backward() before the next forward / optimizer step")

    # ---- direct-gradient backward passes (flat buffers): one chain rule for all paths, one join of the side streams
    def set_deferred(self, on):
        if on == self._deferred:
            return
        if self._pending is not None:
            self.finish_backward()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.srg_set_deferred_chain(self.h, int(on), self.stream()))
            if on:
                torch.cuda.current_stream(self.device).synchronize()   # one-off: the cleared accumulators are visible to all streams
        self._deferred = on

    def backward_begin(self, grads):
        """First direct-mode backward call of an autograd pass: defer the chain rule through the folded message weights
        and have the autograd engine call finish_backward() when the whole pass has been queued."""
        self.set_deferred(True)
        task = torch._C._current_graph_task_id()
        if self._pending is not None and self._pending["task"] != task:
            self.finish_backward()      # an earlier pass died before its callback ran: settle it first
        if self._pending is None:
            self._pending = {"grads": grads, "events": [], "task": task}
            torch.autograd.Variable._execution_engine.queue_callback(self.finish_backward)

    def backward_mark(self):
        """Record the end of one path's backward kernels on the stream they were queued on."""
        k = len(self._pending["events"])
        if k >= len(self._events):
            self._events.append(torch.cuda.Event())
        ev = self._events[k]
        ev.record(torch.cuda.current_stream(self.device))
        self._pending["events"].append(ev)

    def finish_backward(self):
        """Runs on the stream that called backward(): wait for every path (they may have run on side streams -- autograd
        does not join streams of functions that return no gradients), then apply the chain rule once."""
        pend, self._pending = self._pending, None
        if pend is None:
            return
        with torch.cuda.device(self.device):
            cur = torch.cuda.current_stream(self.device)
            for ev in pend["events"]:
                cur.wait_event(ev)
            sg = _grad_struct(pend["grads"], self)
            _lib.check(self.lib.srg_chain_finalize(self.h, ctypes.byref(sg), self.stream()))

    def stream(self):
        """Current stream of THIS engine's device (the caller's current device may be another GPU)."""
        return _lib.stream_ptr(self.device)

    def workspace(self, mode, B, prec, save, k=None, nbest=None):
        """Uninitialised device workspace of one call; k: srg_situation_nouns on B images x k candidate verbs, and
        with nbest: srg_situation_nbest of the `nbest` best situations over k candidate verbs."""
        if k is None:
            n = self.lib.srg_workspace_bytes(self.h, mode, B, prec, int(save))
        elif nbest is None:
            n = self.lib.srg_situation_workspace_bytes(self.h, B, k, prec)
        else:
            n = self.lib.srg_situation_nbest_workspace_bytes(self.h, B, k, nbest, prec)
        ws = torch.empty(n, dtype=torch.uint8, device=self.device)
        if _POISON_WS:      # tests: every byte 0xFF = NaN as fp32 / bf16, -1 as int32: a read of a workspace location
            ws.fill_(0xFF)  # nobody wrote shows up as NaN in the results instead of hiding behind fresh (zeroed) memory
        return ws


def _stats_view(eng, ws, mode, B, prec, save):
    """(workspace tensor, device pointer) of the per-tile softmax statistics the classifier GEMM left in `ws`."""
    off = eng.lib.srg_workspace_stats_offset(eng.h, mode, B, prec, int(save), _lib.ptr(ws))
    return ws, ws.data_ptr() + off


def _prec_code(name):
    if name in ("bf16", SRG_PREC_BF16):
        return SRG_PREC_BF16
    if name in ("fp32", SRG_PREC_FP32):
        return SRG_PREC_FP32
    raise ValueError("precision must be 'bf16' or 'fp32'")


def _as_feat(x, D):
    if not x.is_cuda:
        raise _lib.SrgError("the GGNN stage has no CPU path: features must be CUDA tensors")
    x = x.reshape(x.shape[0], -1)
    if x.shape[1] != D:
        raise _lib.SrgError("backbone features have %d channels, expected %d" % (x.shape[1], D))
    return x.float().contiguous()     # keeps the autograd graph: the stages return dL/dfeat when it is needed


def _grad_struct(named, engine):
    """Zero-initialised fp32 gradient buffers + the srg_grads struct pointing at them."""
    fields = {}
    for n in _lib._PARAM_FIELDS + ["role_emb", "verb_emb"]:
        t = named.get(n)
        fields[n] = ctypes.c_void_p(t.data_ptr()) if t is not None else None
    return _lib.SrgGrads(**fields)


_GGNN_FIELDS = _lib._PARAM_FIELDS[:14]


class _GradTap:
    """Where the loss kernels put d(loss)/d(logits) for a stage that is waiting for it: the bf16, zero-padded operand
    buffer of the classifier's backward GEMMs inside the stage's workspace.  `FCGGNN.verb_loss` / `nouns_loss` write
    there directly when they are applied to the very tensor a `predict_*` call returned, so the fp32 gradient tensor is
    never materialised (nor re-read and converted).  autograd still orders the two nodes: the stage returns a 1-element
    `tap` tensor next to the logits, the loss takes it as an input and hands back a (dummy) gradient for it."""

    def __init__(self, ws, ptr):
        self.ws, self.ptr, self.written = ws, ptr, False


class _NounsStage(torch.autograd.Function):
    """predict_nouns minus the backbone (model.py:117-155).  Input 2 is the fp32 [B, D] feature tensor; its gradient is
    returned when it requires grad (and only then: otherwise the backward passes dfeat = NULL)."""

    @staticmethod
    def forward(ctx, model, grad_on, feat, verb, keep, seed, slot, role_emb, verb_emb, *params):
        eng = model._engine_for(feat.device)
        prec = _prec_code(model.precision)
        B = feat.shape[0]
        need_grad = grad_on and any(ctx.needs_input_grad)
        if need_grad and prec != SRG_PREC_BF16:
            raise _lib.SrgError("precision='fp32' is a forward-only parity mode; use torch.no_grad() or precision='bf16'")
        eng.ensure_packed(model, prec)
        drop_p = model.drop_p if (keep is not None or seed is not None) else 0.0
        logits = torch.empty(B * eng.R, eng.Lpad, dtype=torch.float32, device=feat.device)
        ws = eng.workspace(SRG_MODE_NOUN, B, prec, need_grad)
        verb = verb.detach().to(torch.int64).contiguous()
        _lib.check(eng.lib.srg_nouns_forward(eng.h, _lib.ptr(feat), _lib.ptr(verb), B, _lib.ptr(role_emb),
                                             _lib.ptr(verb_emb), _lib.ptr(keep), drop_p, _lib.ptr(seed), slot,
                                             _lib.ptr(logits), eng.Lpad, prec, int(need_grad), _lib.ptr(ws), ws.numel(),
                                             eng.stream()))
        if need_grad:
            ctx.eng, ctx.ws, ctx.B, ctx.drop_p, ctx.slot = eng, ws, B, drop_p, slot
            ctx.pack_gen = eng.pack_gen
            ctx.direct = model._direct_grads()
            ctx.live = (role_emb, verb_emb) + tuple(params)       # the Parameter objects (for .grad in direct mode)
            ctx.save_for_backward(feat, verb, keep, seed, role_emb, verb_emb, *params)
            ctx.side = _GradTap(ws, ws.data_ptr() + eng.lib.srg_workspace_dlogits_offset(eng.h, SRG_MODE_NOUN, B,
                                                                                        _lib.ptr(ws)))
            ctx.set_materialize_grads(False)
        model._last_stats = _stats_view(eng, ws, SRG_MODE_NOUN, B, prec, need_grad)
        model._last_side = ctx.side if need_grad else None
        return logits.view(B, eng.R, eng.Lpad)[:, :, :eng.L], torch.zeros(1, dtype=torch.float32, device=feat.device)

    @staticmethod
    def backward(ctx, dlogits, dtap):
        eng = ctx.eng
        names = ["role_emb", "verb_emb"] + _GGNN_FIELDS + ["Wc_noun", "bc_noun"]
        in_ws, ctx.side.written = ctx.side.written, False
        if dlogits is None and not in_ws:           # nothing downstream produced a gradient for these logits
            return (None,) * (7 + len(names))
        eng.check_pack_gen(ctx.pack_gen)
        feat, verb, keep, seed, role_emb, verb_emb, *params = ctx.saved_tensors
        B = ctx.B
        dl, ldl = (None, eng.Lpad) if dlogits is None else _padded_grad(dlogits.reshape(B * eng.R, eng.L), eng.Lpad)
        if ctx.direct:   # flat-buffer mode: the kernels accumulate straight into the (pre-zeroed) .grad views
            grads = {n: p.grad for n, p in zip(names, ctx.live)}
            eng.backward_begin(grads)
        else:
            grads = {n: torch.zeros_like(p) for n, p in zip(names, (role_emb, verb_emb) + tuple(params))}
            eng.set_deferred(False)
        sg = _grad_struct(grads, eng)
        dfeat = torch.empty_like(feat) if ctx.needs_input_grad[2] else None
        _lib.check(eng.lib.srg_nouns_backward_feat(eng.h, _lib.ptr(dl), ldl, int(in_ws), _lib.ptr(feat), _lib.ptr(verb),
                                                   B, _lib.ptr(role_emb), _lib.ptr(verb_emb), _lib.ptr(keep),
                                                   ctx.drop_p, _lib.ptr(seed), ctx.slot, ctypes.byref(sg),
                                                   _lib.ptr(dfeat), _lib.ptr(ctx.ws), ctx.ws.numel(), eng.stream()))
        ctx.ws = None
        if ctx.direct:
            eng.backward_mark()
            return (None, None, dfeat) + (None,) * (4 + len(names))
        out = [grads[n] for n in _GGNN_FIELDS + ["Wc_noun", "bc_noun"]]
        return (None, None, dfeat, None, None, None, None, grads["role_emb"], grads["verb_emb"], *out)


class _VerbStage(torch.autograd.Function):
    """predict_verb minus the backbone (model.py:160-168); dL/dfeat for input 2 as in _NounsStage."""

    @staticmethod
    def forward(ctx, model, grad_on, feat, keep, seed, slot, *params):
        eng = model._engine_for(feat.device)
        prec = _prec_code(model.precision)
        B = feat.shape[0]
        need_grad = grad_on and any(ctx.needs_input_grad)
        if need_grad and prec != SRG_PREC_BF16:
            raise _lib.SrgError("precision='fp32' is a forward-only parity mode; use torch.no_grad() or precision='bf16'")
        eng.ensure_packed(model, prec)
        drop_p = model.drop_p if (keep is not None or seed is not None) else 0.0
        logits = torch.empty(B, eng.Vpad, dtype=torch.float32, device=feat.device)
        ws = eng.workspace(SRG_MODE_VERB, B, prec, need_grad)
        _lib.check(eng.lib.srg_verb_forward(eng.h, _lib.ptr(feat), B, _lib.ptr(keep), drop_p, _lib.ptr(seed), slot,
                                            _lib.ptr(logits), eng.Vpad, prec, int(need_grad), _lib.ptr(ws), ws.numel(),
                                            eng.stream()))
        if need_grad:
            ctx.eng, ctx.ws, ctx.B, ctx.drop_p, ctx.slot = eng, ws, B, drop_p, slot
            ctx.pack_gen = eng.pack_gen
            ctx.direct = model._direct_grads()
            ctx.live = tuple(params)
            ctx.save_for_backward(keep, seed, *params)
            ctx.side = _GradTap(ws, ws.data_ptr() + eng.lib.srg_workspace_dlogits_offset(eng.h, SRG_MODE_VERB, B,
                                                                                        _lib.ptr(ws)))
            ctx.set_materialize_grads(False)
        model._last_stats = _stats_view(eng, ws, SRG_MODE_VERB, B, prec, need_grad)
        model._last_side = ctx.side if need_grad else None
        return logits[:, :eng.V], torch.zeros(1, dtype=torch.float32, device=feat.device)

    @staticmethod
    def backward(ctx, dlogits, dtap):
        eng = ctx.eng
        names = _GGNN_FIELDS + ["Wc_verb", "bc_verb"]
        in_ws, ctx.side.written = ctx.side.written, False
        if dlogits is None and not in_ws:
            return (None,) * (6 + len(names))
        eng.check_pack_gen(ctx.pack_gen)
        keep, seed, *params = ctx.saved_tensors
        B = ctx.B
        dl, ldl = (None, eng.Vpad) if dlogits is None else _padded_grad(dlogits.reshape(B, eng.V), eng.Vpad)
        if ctx.direct:
            grads = {n: p.grad for n, p in zip(names, ctx.live)}
            eng.backward_begin(grads)
        else:
            grads = {n: torch.zeros_like(p) for n, p in zip(names, params)}
            eng.set_deferred(False)
        sg = _grad_struct(grads, eng)
        dfeat = torch.empty(B, eng.D, dtype=torch.float32, device=eng.device) if ctx.needs_input_grad[2] else None
        _lib.check(eng.lib.srg_verb_backward_feat(eng.h, _lib.ptr(dl), ldl, int(in_ws), B, _lib.ptr(keep), ctx.drop_p,
                                                  _lib.ptr(seed), ctx.slot, ctypes.byref(sg), _lib.ptr(dfeat),
                                                  _lib.ptr(ctx.ws), ctx.ws.numel(), eng.stream()))
        ctx.ws = None
        if ctx.direct:
            eng.backward_mark()
            return (None, None, dfeat) + (None,) * (3 + len(names))
        return (None, None, dfeat, None, None, None, *[grads[n] for n in names])


class _GGSNNStage(torch.autograd.Function):
    """GGSNN.forward (model.py:59-86) on caller-supplied node states and mask, with its backward (bf16 only).
    hidden: [B*R, D] (or [B, R, D]) with mask [B, R, R], or [B, D] with mask None (verb node)."""

    @staticmethod
    def forward(ctx, model, hidden, mask, *params):
        eng = model._engine_for(hidden.device)
        eng.ensure_packed(model, SRG_PREC_BF16)
        h, mode, B, mk = _ggsnn_inputs(eng, hidden, mask, mask is None)
        ws = eng.workspace(mode, B, SRG_PREC_BF16, True)
        _lib.check(eng.lib.srg_ggnn_forward(eng.h, mode, _lib.ptr(h), _lib.ptr(mk), B, SRG_PREC_BF16, 1, _lib.ptr(ws),
                                            ws.numel(), eng.stream()))
        ctx.eng, ctx.ws, ctx.B, ctx.mode = eng, ws, B, mode
        ctx.pack_gen = eng.pack_gen
        ctx.direct = model._direct_grads()
        ctx.live = tuple(params)          # the Parameter objects (for .grad in direct mode)
        ctx.in_shape, ctx.in_dtype = hidden.shape, hidden.dtype
        ctx.mask_meta = None if mask is None else (mask.device, mask.dtype)
        ctx.save_for_backward(mk, *params)
        return h

    @staticmethod
    def backward(ctx, dout):
        eng = ctx.eng
        eng.check_pack_gen(ctx.pack_gen)
        mk, *params = ctx.saved_tensors
        g = dout.detach().to(torch.float32).contiguous()
        if ctx.direct:   # flat-buffer mode: the kernels accumulate straight into the (pre-zeroed) .grad views
            grads = {n: p.grad for n, p in zip(_GGNN_FIELDS, ctx.live)}
            eng.backward_begin(grads)
        else:
            grads = {n: torch.zeros_like(p) if ctx.needs_input_grad[3 + i] else None
                     for i, (n, p) in enumerate(zip(_GGNN_FIELDS, params))}
            eng.set_deferred(False)
        dh = torch.empty_like(g) if ctx.needs_input_grad[1] else None
        dm = torch.empty_like(mk) if ctx.needs_input_grad[2] else None     # no dL/dmask pass unless it is wanted
        sg = _grad_struct(grads, eng)
        _lib.check(eng.lib.srg_ggnn_backward(eng.h, ctx.mode, _lib.ptr(g), _lib.ptr(mk), _lib.ptr(dm), _lib.ptr(dh),
                                             ctx.B, ctypes.byref(sg), _lib.ptr(ctx.ws), ctx.ws.numel(), eng.stream()))
        ctx.ws = None
        if ctx.direct:
            eng.backward_mark()
        dh = None if dh is None else dh.view(ctx.in_shape).to(ctx.in_dtype)
        dm = None if dm is None else dm.to(*ctx.mask_meta)
        return (None, dh, dm, *[None if ctx.direct else grads[n] for n in _GGNN_FIELDS])


def _ggsnn_inputs(eng, hidden, mask, verb):
    """(fp32 [rows, D] copy of the states, mode, B, fp32 [B, R, R] mask or None) for srg_ggnn_forward."""
    h = hidden.detach().float().contiguous().clone()
    if verb:
        B, mode, mk = h.shape[0], SRG_MODE_VERB, None
        rows = B
    else:
        B, mode = mask.shape[0], SRG_MODE_NOUN
        mk = mask.detach().to(device=h.device, dtype=torch.float32).contiguous()
        rows = B * eng.R
        if tuple(mk.shape) != (B, eng.R, eng.R):
            raise _lib.SrgError("mask must be [B, %d, %d], got %s" % (eng.R, eng.R, tuple(mask.shape)))
    if h.numel() != rows * eng.D:
        raise _lib.SrgError("hidden_state has %d elements, expected %d rows of %d" % (h.numel(), rows, eng.D))
    return h, mode, B, mk


def _padded_grad(g, npad):
    """fp32 [rows, n] gradient with unit column stride and a 16-byte aligned row pitch (no copy when the autograd
    engine hands back the padded view produced by the loss kernels)."""
    if g.dtype == torch.float32 and g.dim() == 2 and g.stride(1) == 1 and g.stride(0) >= g.shape[1] and \
            g.stride(0) % 4 == 0 and g.data_ptr() % 16 == 0:
        return g, g.stride(0)
    buf = torch.zeros(g.shape[0], npad, dtype=torch.float32, device=g.device)
    buf[:, :g.shape[1]] = g
    return buf, npad


def _rows_view(logits, n):
    """[rows, n] view with unit column stride of a [..., n] logits tensor, and its leading dimension."""
    x = logits
    if x.dtype != torch.float32:
        x = x.float()
    lead = x.shape[:-1]
    ok = x.stride(-1) == 1
    ld = x.stride(-2) if x.dim() >= 2 else n
    if ok and x.dim() == 3:
        ok = x.stride(0) == x.shape[1] * ld
    if not ok or ld < n:
        x = x.contiguous()
        ld = n
    rows = 1
    for s in lead:
        rows *= s
    return x, rows, ld


class _LossOpts:
    """Validated `weight` / `label_smoothing` / `reduction` of one verb_loss / nouns_loss call (torch's
    F.cross_entropy keywords), or None from `make` when all three hold their defaults: the loss then runs the
    default-option kernels, launch for launch.  Everything is checked here, before any engine call."""

    def __init__(self, weight, eps, reduction):
        self.weight, self.eps, self.reduction = weight, eps, reduction
        self.red = _lib.SRG_REDUCTION[reduction]
        # the denominators' cache key: a new weight tensor, or an in-place change of this one, is never stale
        self.wkey = None if weight is None else (weight.data_ptr(), weight._version)

    @staticmethod
    def make(weight, label_smoothing, reduction, n_classes, device, what):
        if reduction not in _lib.SRG_REDUCTION:
            raise ValueError("%s: reduction must be 'mean', 'sum' or 'none', got %r" % (what, reduction))
        eps = float(label_smoothing)
        if not 0.0 <= eps <= 1.0:
            raise ValueError("%s: label_smoothing must be in [0, 1], got %r" % (what, label_smoothing))
        if weight is not None:
            if not isinstance(weight, torch.Tensor):
                raise _lib.SrgError("%s: weight must be a tensor, got %s" % (what, type(weight).__name__))
            if weight.requires_grad:
                raise _lib.SrgError("%s: weight is data and must not require grad (pass weight.detach())" % what)
            if weight.dim() != 1 or weight.numel() != n_classes:
                raise _lib.SrgError("%s: weight must have shape [%d], got %s" % (what, n_classes, tuple(weight.shape)))
            if weight.dtype != torch.float32:
                raise _lib.SrgError("%s: weight must be float32, got %s" % (what, weight.dtype))
            if weight.device != device:
                raise _lib.SrgError("%s: weight is on %s, the logits on %s" % (what, weight.device, device))
        if weight is None and eps == 0.0 and reduction == "mean":
            return None
        return _LossOpts(None if weight is None else weight.contiguous(), eps, reduction)

    def struct(self, per_target=None, grad_per_target=None):
        return _lib.SrgLossOpts(_lib.ptr(self.weight), self.eps, self.red, _lib.ptr(per_target),
                                _lib.ptr(grad_per_target))


class _NounsLoss(torch.autograd.Function):
    """FCGGNN.nouns_loss (model.py:189-201).  Forward only reads what the loss needs (with the classifier's per-tile
    softmax statistics: the three target logits of a row); the gradient is produced in backward, already multiplied by
    the incoming d(loss), in one pass over the logits.  opts (_LossOpts or None): class weights, label smoothing and
    the reduction; with "none" the loss is [B, 3, R] and backward takes any upstream gradient of that shape."""

    @staticmethod
    def forward(ctx, model, grad_on, logits, gt_nouns, stats, tap, side, opts):
        eng = model._engine_for(logits.device)
        x, rows, ld = _rows_view(logits, eng.L)
        if x.data_ptr() != logits.data_ptr():
            stats = side = None                    # the logits were copied / converted: neither applies
        B = rows // eng.R
        gt = gt_nouns.detach().to(torch.int64).contiguous()
        counts = None
        if opts is None or opts.red == _lib.SRG_REDUCTION["mean"]:
            # the denominators depend on the targets (and the class weights) only: nouns_loss(pred_nouns, gt) and
            # nouns_loss(gt_pred_nouns, gt) of one step (sr.py:69-70) share them, which also halves the small
            # all-reduces of a sharded step
            wkey = None if opts is None else opts.wkey
            key = (gt.data_ptr(), gt._version, tuple(gt.shape), torch.cuda.current_stream(gt.device).cuda_stream, wkey)
            cached = model._counts_cache
            if cached is not None and cached[0] == key:
                counts = cached[1]
            else:
                counts = torch.empty(3, dtype=torch.float32, device=logits.device)
                if wkey is None:
                    _lib.check(eng.lib.srg_count_targets(eng.h, _lib.ptr(gt), B, _lib.ptr(counts), eng.stream()))
                else:
                    _lib.check(eng.lib.srg_count_targets_weighted(eng.h, _lib.ptr(gt), B, _lib.ptr(opts.weight),
                                                                  _lib.ptr(counts), eng.stream()))
                if model.loss_group is not None:
                    torch.distributed.all_reduce(counts, group=model.loss_group)
                # holding gt (and the weight) keeps their addresses from being reused
                model._counts_cache = (key, counts, gt, None if opts is None else opts.weight)
        st = ctypes.c_void_p(stats[1]) if stats else None
        if opts is None:
            loss = torch.zeros((), dtype=torch.float32, device=logits.device)
            _lib.check(eng.lib.srg_nouns_loss(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), B, _lib.ptr(counts),
                                              _lib.ptr(loss), None, 1.0, st, eng.stream()))
        elif opts.reduction == "none":
            loss = torch.empty(B, 3, eng.R, dtype=torch.float32, device=logits.device)
            _lib.check(eng.lib.srg_nouns_loss_ex(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), B, _lib.ptr(counts), None, None,
                                                 1.0, st, ctypes.byref(opts.struct(per_target=loss)), eng.stream()))
        else:   # the per-target terms are summed in a fixed order: bit-identical losses from call to call
            loss = torch.zeros((), dtype=torch.float32, device=logits.device)
            terms = torch.empty(B * 3 * eng.R, dtype=torch.float32, device=logits.device)
            _lib.check(eng.lib.srg_nouns_loss_ex(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), B, _lib.ptr(counts),
                                                 _lib.ptr(loss), None, 1.0, st,
                                                 ctypes.byref(opts.struct(per_target=terms)), eng.stream()))
        if grad_on and (ctx.needs_input_grad[2] or ctx.needs_input_grad[5]):
            ctx.save_for_backward(x, gt, counts)
            ctx.eng, ctx.geom, ctx.shape, ctx.stats, ctx.opts = eng, (rows, ld, B), tuple(logits.shape), stats, opts
            ctx.side = side if (side is not None and ctx.needs_input_grad[5] and ld == eng.Lpad) else None
        return loss

    @staticmethod
    def backward(ctx, gout):
        x, gt, counts = ctx.saved_tensors
        eng, (rows, ld, B), stats, side, opts = ctx.eng, ctx.geom, ctx.stats, ctx.side, ctx.opts
        gout = gout.detach().to(torch.float32).contiguous()
        st = ctypes.c_void_p(stats[1]) if stats else None
        ctx.stats = None
        per_target = opts is not None and opts.reduction == "none"
        o = None if opts is None else ctypes.byref(opts.struct(grad_per_target=gout if per_target else None))
        gscale = None if per_target else _lib.ptr(gout)
        if side is not None:     # straight into the stage's bf16 operand buffer; the tap carries the dependency
            _lib.check(eng.lib.srg_nouns_loss_backward_ex(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), B, _lib.ptr(counts),
                                                          gscale, 1.0, None, ctypes.c_void_p(side.ptr),
                                                          int(side.written), st, o, eng.stream()))
            side.written = True
            return None, None, None, None, None, gout.new_zeros(1), None, None
        dl = torch.empty(rows, ld, dtype=torch.float32, device=x.device)
        _lib.check(eng.lib.srg_nouns_loss_backward_ex(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), B, _lib.ptr(counts),
                                                      gscale, 1.0, _lib.ptr(dl), None, 0, st, o, eng.stream()))
        return None, None, dl[:, :eng.L].view(ctx.shape), None, None, None, None, None


class _VerbLoss(torch.autograd.Function):
    """FCGGNN.verb_loss (model.py:182-187); same split between forward and backward, and the same options, as
    _NounsLoss ("none": a [B] loss)."""

    @staticmethod
    def forward(ctx, model, grad_on, logits, gt_verb, stats, tap, side, opts):
        eng = model._engine_for(logits.device)
        x, rows, ld = _rows_view(logits, eng.V)
        if x.data_ptr() != logits.data_ptr():
            stats = side = None
        gt = gt_verb.detach().to(torch.int64).contiguous()
        # The mean is over the GLOBAL batch (the reference computes the loss on the gathered logits of all replicas,
        # sr.py:66-68).  Shards may be unequal (tail batch of an epoch), so rows * world is NOT the denominator: the
        # caller states the global batch (model.global_batch), or the local batch sizes are all-reduced on the stream.
        # With class weights the denominator is the global sum of the targets' weights, which only the all-reduce of
        # the local sums gives.
        inv, total = 1.0 / rows, None
        if opts is not None and opts.weight is not None and opts.red == _lib.SRG_REDUCTION["mean"]:
            total = torch.empty(1, dtype=torch.float32, device=logits.device)
            _lib.check(eng.lib.srg_verb_weight_total(eng.h, _lib.ptr(gt), rows, _lib.ptr(opts.weight),
                                                     _lib.ptr(total), eng.stream()))
            if model.loss_group is not None:
                torch.distributed.all_reduce(total, group=model.loss_group)
        elif model.loss_group is not None and (opts is None or opts.red == _lib.SRG_REDUCTION["mean"]):
            if model.global_batch is not None:
                inv = 1.0 / float(model.global_batch)
            else:
                total = torch.full((1,), float(rows), dtype=torch.float32, device=logits.device)
                torch.distributed.all_reduce(total, group=model.loss_group)
        st = ctypes.c_void_p(stats[1]) if stats else None
        if opts is None:
            loss = torch.zeros((), dtype=torch.float32, device=logits.device)
            _lib.check(eng.lib.srg_verb_loss(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), rows, inv, _lib.ptr(total),
                                             _lib.ptr(loss), None, 1.0, st, eng.stream()))
        elif opts.reduction == "none":
            loss = torch.empty(rows, dtype=torch.float32, device=logits.device)
            _lib.check(eng.lib.srg_verb_loss_ex(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), rows, inv, _lib.ptr(total), None,
                                                None, 1.0, st, ctypes.byref(opts.struct(per_target=loss)),
                                                eng.stream()))
        else:
            loss = torch.zeros((), dtype=torch.float32, device=logits.device)
            terms = torch.empty(rows, dtype=torch.float32, device=logits.device)
            _lib.check(eng.lib.srg_verb_loss_ex(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), rows, inv, _lib.ptr(total),
                                                _lib.ptr(loss), None, 1.0, st,
                                                ctypes.byref(opts.struct(per_target=terms)), eng.stream()))
        if grad_on and (ctx.needs_input_grad[2] or ctx.needs_input_grad[5]):
            saved = (x, gt) if total is None else (x, gt, total)
            ctx.save_for_backward(*saved)
            ctx.eng, ctx.geom, ctx.shape, ctx.stats, ctx.opts = eng, (rows, ld, inv), tuple(logits.shape), stats, opts
            ctx.side = side if (side is not None and ctx.needs_input_grad[5] and ld == eng.Vpad) else None
        return loss

    @staticmethod
    def backward(ctx, gout):
        x, gt, *rest = ctx.saved_tensors
        total = rest[0] if rest else None
        eng, (rows, ld, inv), stats, side, opts = ctx.eng, ctx.geom, ctx.stats, ctx.side, ctx.opts
        gout = gout.detach().to(torch.float32).contiguous()
        st = ctypes.c_void_p(stats[1]) if stats else None
        ctx.stats = None
        per_target = opts is not None and opts.reduction == "none"
        o = None if opts is None else ctypes.byref(opts.struct(grad_per_target=gout if per_target else None))
        gscale = None if per_target else _lib.ptr(gout)
        if side is not None:
            _lib.check(eng.lib.srg_verb_loss_backward_ex(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), rows, inv,
                                                         _lib.ptr(total), gscale, 1.0, None, ctypes.c_void_p(side.ptr),
                                                         int(side.written), st, o, eng.stream()))
            side.written = True
            return None, None, None, None, None, gout.new_zeros(1), None, None
        dl = torch.empty(rows, ld, dtype=torch.float32, device=x.device)
        _lib.check(eng.lib.srg_verb_loss_backward_ex(eng.h, _lib.ptr(x), ld, _lib.ptr(gt), rows, inv, _lib.ptr(total),
                                                     gscale, 1.0, _lib.ptr(dl), None, 0, st, o, eng.stream()))
        return None, None, dl[:, :eng.V].view(ctx.shape), None, None, None, None, None


def _has_batchnorm_in_train(module):
    """A backbone whose BatchNorm layers are in training mode updates its running statistics on every call; calling
    it once instead of twice would change those statistics, so the dedupe is skipped in that case."""
    return any(isinstance(m, nn.modules.batchnorm._BatchNorm) and m.training for m in module.modules())


class GGSNN(nn.Module):
    """Parameter container + drop-in forward of the reference's GGSNN (model.py:38-86)."""

    def __init__(self, layersize):
        super().__init__()
        self.W_p = nn.Linear(layersize, layersize)
        self.W_z = nn.Linear(layersize, layersize)
        self.U_z = nn.Linear(layersize, layersize)
        self.W_r = nn.Linear(layersize, layersize)
        self.U_r = nn.Linear(layersize, layersize)
        self.W_h = nn.Linear(layersize, layersize)
        self.U_h = nn.Linear(layersize, layersize)
        self._owner = None

    def forward(self, hidden_state, mask=None, verb=False):
        """model.py:59-86 with the reference signature: hidden_state [B*R, D] with mask [B, R, R] (role graph), or
        [B, D] with verb=True (verb node).  Differentiable in bf16 precision: when grad is enabled and hidden_state, mask
        or a GGSNN parameter requires grad, the CUDA backward returns the gradients of all three (dL/dmask only when
        mask.requires_grad).  precision='fp32' is forward-only and raises when a gradient is needed."""
        owner = self._owner() if self._owner is not None else None
        if owner is None:
            raise _lib.SrgError("GGSNN.forward needs the owning FCGGNN (it holds the CUDA engine)")
        return owner._ggsnn_forward(hidden_state, mask, verb)


class FCGGNN(nn.Module):
    def __init__(self, encoder, D_hidden_state, backbone="resnet152", precision="bf16", pretrained=None):
        super().__init__()
        self.encoder = encoder
        self.D = D_hidden_state
        self.precision = precision
        self.drop_p = 0.5
        self.loss_group = None          # torch.distributed group over which loss denominators are global
        self.global_batch = None        # images of the current GLOBAL batch when the caller knows it (saves the
                                        # all-reduce of the local batch sizes in verb_loss); None = all-reduce
        self.dropout_masks = None       # optional (verb, pred-noun, gt-noun) uint8 keep-masks for parity tests
        self._seed_state = {}           # device -> int64[1] dropout seed counter (Philox key of the next forward)
        self._step_seed = None          # seed shared by the three paths of the forward() call in flight
        self.last_drop_seed = None      # seed tensor the most recent training forward used (tests replay its masks)
        self.role_emb = nn.Embedding(encoder.get_num_roles() + 1, D_hidden_state, padding_idx=encoder.get_num_roles())
        self.verb_emb = nn.Embedding(encoder.get_num_verbs(), D_hidden_state)
        if backbone == "resnet152":
            self.convnet_verbs = resnet(encoder.get_num_verbs(), pretrained)
            self.convnet_nouns = resnet(encoder.get_num_labels(), pretrained)
        else:  # GGNN-stage benchmarks / tests: `img` already holds the [B, D] backbone features
            self.convnet_verbs = nn.Identity()
            self.convnet_nouns = nn.Identity()
        self.ggsnn = GGSNN(layersize=D_hidden_state)
        self.verb_classifier = nn.Sequential(nn.Dropout(self.drop_p), nn.Linear(D_hidden_state, encoder.get_num_verbs()))
        self.nouns_classifier = nn.Sequential(nn.Dropout(self.drop_p), nn.Linear(D_hidden_state, encoder.get_num_labels()))
        import weakref
        self.ggsnn._owner = weakref.ref(self)
        self._engines = {}
        self._side_streams = {}
        self.overlap_streams = True      # run the verb path on a side stream (see forward)
        self._flat = None                # parallel.attach(): flat gradient / parameter buffers
        self._last_stats = None
        self._last_side = None
        self._counts_cache = None        # (key, counts, targets, weight) of the last nouns_loss call

    # sr.py accesses model.module.* when CUDA is available (DataParallel wrapper in the reference)
    @property
    def module(self):
        return self

    def _engine_for(self, device):
        key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
        eng = self._engines.get(key)
        if eng is None:
            eng = _Engine(self, torch.device("cuda", key[1]))
            self._engines[key] = eng
        return eng

    def _direct_grads(self):
        """True when parallel.attach() installed flat gradient buffers: the backward kernels then accumulate into the
        pre-zeroed `.grad` views directly (no per-tensor zero-fill and no autograd accumulation kernels)."""
        flat = self._flat
        if flat is None:
            return False
        return all(p.grad is not None and p.grad.dtype == torch.float32 and p.grad.is_contiguous() for p in flat.params)

    def _ggnn_params(self):
        g = self.ggsnn
        return [g.W_p.weight, g.W_p.bias, g.W_z.weight, g.W_z.bias, g.U_z.weight, g.U_z.bias, g.W_r.weight, g.W_r.bias,
                g.U_r.weight, g.U_r.bias, g.W_h.weight, g.W_h.bias, g.U_h.weight, g.U_h.bias]

    def _draw_seed(self, device):
        """A fresh dropout seed (device int64[1]) without a host synchronisation, so that it also works inside a CUDA
        graph: the seed tensor handed out is a copy of a device counter that is then advanced.  The counter starts from
        torch's CPU generator, so `torch.manual_seed` makes training runs repeatable."""
        state = self._seed_state.get(device)
        if state is None:
            state = torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).to(device)
            self._seed_state[device] = state
        seed = state.clone()
        state.add_(1)
        self.last_drop_seed = seed
        return seed

    def _dropout(self, which, device):
        """(explicit keep-mask | None, Philox seed | None) for path `which` (0 verb, 1 predicted-verb nouns, 2 gt nouns).
        Eval mode: (None, None).  model.py:106,110: nn.Dropout(0.5) in front of both classifiers."""
        if not self.training:
            return None, None
        if self.dropout_masks is not None:
            m = self.dropout_masks[which]
            return (None if m is None else m.to(device=device, dtype=torch.uint8).contiguous()), None
        return None, (self._step_seed if self._step_seed is not None else self._draw_seed(device))

    def dropout_mask(self, which, rows, seed=None):
        """The uint8 keep-mask [rows, D] the Philox path applied (applies) on path `which` for `seed` (default: the
        seed of the most recent training forward).  Test helper: lets the oracle replay a training step's dropout."""
        seed = self.last_drop_seed if seed is None else seed
        eng = self._engine_for(seed.device)
        out = torch.empty(rows, self.D, dtype=torch.uint8, device=seed.device)
        _lib.check(eng.lib.srg_dropout_mask(_lib.ptr(seed), which, self.drop_p, rows, self.D, _lib.ptr(out), eng.stream()))
        return out

    # ---- reference API -------------------------------------------------------------------------
    def predict_nouns(self, img, gt_verb, batch_size, _mask_slot=1, _feat=None):
        # `_feat`: backbone features computed once by forward() for both noun passes (the reference runs the
        # convnet_nouns twice on the same images, model.py:116,176-178)
        feat = _feat if _feat is not None else _as_feat(self.convnet_nouns(img), self.D)
        if feat.shape[0] != batch_size:
            raise _lib.SrgError("batch_size %d does not match the features (%d)" % (batch_size, feat.shape[0]))
        keep, seed = self._dropout(_mask_slot, feat.device)
        gt_verb = gt_verb.to(feat.device)
        out, tap = _NounsStage.apply(self, torch.is_grad_enabled(), feat, gt_verb, keep, seed, _mask_slot,
                                     self.role_emb.weight, self.verb_emb.weight, *self._ggnn_params(),
                                     self.nouns_classifier[1].weight, self.nouns_classifier[1].bias)
        out._srg_stats = self._last_stats      # lets nouns_loss() reuse the classifier's per-tile softmax statistics
        out._srg_tap = (tap, self._last_side) if (tap.requires_grad and self._last_side is not None) else None
        return out

    def predict_verb(self, img, batch_size, _feat=None):
        feat = _feat if _feat is not None else _as_feat(self.convnet_verbs(img), self.D)
        if feat.shape[0] != batch_size:
            raise _lib.SrgError("batch_size %d does not match the features (%d)" % (batch_size, feat.shape[0]))
        keep, seed = self._dropout(0, feat.device)
        out, tap = _VerbStage.apply(self, torch.is_grad_enabled(), feat, keep, seed, 0, *self._ggnn_params(),
                                    self.verb_classifier[1].weight, self.verb_classifier[1].bias)
        out._srg_stats = self._last_stats
        out._srg_tap = (tap, self._last_side) if (tap.requires_grad and self._last_side is not None) else None
        return out

    def forward(self, img, gt_verb, img_nouns=None):
        """model.py:171-180.  `img_nouns` (extension) lets benchmarks feed different synthetic features to the verb
        and noun paths, as the two backbones would produce.

        The verb path and the predicted-verb noun path that depends on it run on side streams, concurrently with the
        gt-verb noun path (which depends on neither); autograd replays the same streams, so the verb and the noun
        backward passes overlap as well."""
        batch_size = img.size(0)
        img_n = img if img_nouns is None else img_nouns
        self._step_seed = None
        if self.training and self.dropout_masks is None and img.is_cuda:
            self._step_seed = self._draw_seed(img.device)       # one Philox key for the three paths of this step
        try:
            return self._forward_paths(img, img_n, gt_verb, batch_size)
        finally:
            self._step_seed = None

    def extract_features(self, img, img_nouns=None):
        """The two backbones (model.py:116,159): (feat_verbs, feat_nouns), fp32 [B, D], differentiable when a backbone
        (or the image) requires grad.  With frozen backbones (model.py:17-18, the default) the features of a fixed image
        under a deterministic transform in eval mode never change: `features.FeatureCache` keeps them across epochs
        (SURVEY section 8f, N3).  That cache is wrong for backbones being fine-tuned."""
        img_n = img if img_nouns is None else img_nouns
        return _as_feat(self.convnet_verbs(img), self.D), _as_feat(self.convnet_nouns(img_n), self.D)

    def forward_features(self, feat_verbs, feat_nouns, gt_verb):
        """`forward` on backbone features instead of images: (pred_verb, pred_nouns, gt_pred_nouns).  In bf16 mode the
        features get their gradients when they require grad (one tensor passed as both inputs: the sum of the three
        paths' gradients)."""
        fv, fn = _as_feat(feat_verbs, self.D), _as_feat(feat_nouns, self.D)
        self._step_seed = None
        if self.training and self.dropout_masks is None:
            self._step_seed = self._draw_seed(fv.device)
        try:
            return self._forward_paths(None, None, gt_verb, fv.shape[0], feat_v=fv, feat_n=fn)
        finally:
            self._step_seed = None

    def _forward_paths(self, img, img_n, gt_verb, batch_size, feat_v=None, feat_n=None):
        # the noun backbone is deterministic unless its BatchNorm layers train: evaluate it once for both noun passes
        # (trainable or not: autograd sums the two passes' gradients into the one feature tensor)
        if feat_n is None and img_n.is_cuda and not (self.training and _has_batchnorm_in_train(self.convnet_nouns)):
            feat_n = _as_feat(self.convnet_nouns(img_n), self.D)
        on_cuda = (feat_v if feat_v is not None else img).is_cuda
        if not (self.overlap_streams and on_cuda):
            pred_verb = self.predict_verb(img, batch_size, _feat=feat_v)
            pred_nouns = self.predict_nouns(img_n, torch.argmax(pred_verb, 1), batch_size, _mask_slot=1, _feat=feat_n)
            gt_pred_nouns = self.predict_nouns(img_n, gt_verb, batch_size, _mask_slot=2, _feat=feat_n)
            return pred_verb, pred_nouns, gt_pred_nouns
        dev = (feat_v if feat_v is not None else img).device
        cur = torch.cuda.current_stream(dev)
        # the weights are packed once, before the fork, so all streams see the same operands
        self._engine_for(dev).ensure_packed(self, _prec_code(self.precision))
        sides = self._side_streams.get(dev)
        if sides is None:
            sides = self._side_streams[dev] = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
        side_v, side_p = sides
        # Three chains of dependent launches: the verb node path (B rows), then the predicted-verb role graph that needs
        # its argmax, and -- independent of both -- the gt-verb role graph.  The first two run on side streams while the
        # third runs on the caller's stream: whenever a launch of one chain is down to its last, partly filled wave of
        # tiles, the free SMs take tiles of the other chain's launch (on a 768-image shard a launch is only ~1.2 waves).
        side_v.wait_stream(cur)
        with torch.cuda.stream(side_v):
            pred_verb = self.predict_verb(img, batch_size, _feat=feat_v)
        side_p.wait_stream(side_v)
        with torch.cuda.stream(side_p):
            pred_nouns = self.predict_nouns(img_n, torch.argmax(pred_verb, 1), batch_size, _mask_slot=1, _feat=feat_n)
        gt_pred_nouns = self.predict_nouns(img_n, gt_verb, batch_size, _mask_slot=2, _feat=feat_n)
        cur.wait_stream(side_p)          # side_p waited for side_v: this joins both
        pred_verb.record_stream(side_p)
        pred_verb.record_stream(cur)
        pred_nouns.record_stream(cur)
        return pred_verb, pred_nouns, gt_pred_nouns

    @staticmethod
    def _stats_ptr(logits, expected_rows_stride):
        """(workspace tensor, device pointer) of the classifier's per-tile softmax statistics if `logits` is the very
        tensor a predict_* call of this model returned (same storage, same layout), else None.  The loss node keeps
        the pair, so the workspace outlives it."""
        st = getattr(logits, "_srg_stats", None)
        if st is None or logits.dtype != torch.float32 or logits.stride(-1) != 1 or \
                logits.stride(-2) != expected_rows_stride:
            return None
        return st

    @staticmethod
    def _tap_of(logits, stats):
        """(tap tensor, _GradTap) when `logits` is the very tensor a predict_* call returned in a differentiable
        forward (same condition as for the softmax statistics), else (None, None)."""
        tp = getattr(logits, "_srg_tap", None) if stats is not None else None
        return tp if tp is not None else (None, None)

    def verb_loss(self, pred_verb, gt_verb, weight=None, label_smoothing=0.0, reduction="mean"):
        """CrossEntropy(pred_verb [B, n_verbs], gt_verb [B]) (model.py:182-187) with the keywords of
        F.cross_entropy: class weights [n_verbs] (data: they must not require grad), label smoothing in [0, 1] and the
        reduction ("none" gives the [B] per-image losses).  The mean is over the global batch under `loss_group`,
        weighted: sum of weight[gt_verb] over all ranks.  A zero denominator gives 0 where torch gives NaN."""
        opts = _LossOpts.make(weight, label_smoothing, reduction, self.encoder.get_num_verbs(), pred_verb.device,
                              "verb_loss")
        eng_pad = _pad256(self.encoder.get_num_verbs())
        stats = self._stats_ptr(pred_verb, eng_pad) if pred_verb.dim() == 2 else None
        tap, side = self._tap_of(pred_verb, stats)
        return _VerbLoss.apply(self, torch.is_grad_enabled(), pred_verb, gt_verb.to(pred_verb.device), stats, tap, side,
                               opts)

    def nouns_loss(self, pred_nouns, gt_nouns, weight=None, label_smoothing=0.0, reduction="mean"):
        """Sum over the 3 annotations of CrossEntropy(ignore_index = n_labels) (model.py:189-201), with the keywords
        of F.cross_entropy as verb_loss: weight [n_labels]; "mean" is taken per annotation (denominator: the global
        sum of weight[y] over its non-ignored targets) and summed; "none" gives [B, 3, R] laid out like gt_nouns, 0 on
        ignored targets."""
        opts = _LossOpts.make(weight, label_smoothing, reduction, self.encoder.get_num_labels(), pred_nouns.device,
                              "nouns_loss")
        eng_pad = _pad256(self.encoder.get_num_labels())
        stats = self._stats_ptr(pred_nouns, eng_pad) if pred_nouns.dim() == 3 else None
        tap, side = self._tap_of(pred_nouns, stats)
        return _NounsLoss.apply(self, torch.is_grad_enabled(), pred_nouns, gt_nouns.to(pred_nouns.device), stats, tap,
                                side, opts)

    # ---- top-k situation decode ----------------------------------------------------------------
    @torch.no_grad()
    def situations_from_features(self, feat_verbs, feat_nouns, k=5, verbs=None):
        """The k best situations of each image from the backbone features ([B, D] each): the verb path, the top k
        verbs with their log-softmax, then the role graphs of all B*k (image, verb) pairs in one call (the node init
        reads each image's feature row k times instead of copying it) and the top-1 label of every role slot.
        verbs ([B, k'] int64, optional): decode these candidate verbs instead (feat_verbs is then not used and may be
        None; verb_logp is None and the score is the label term only) -- e.g. `verbs=gt_verb[:, None]` for the
        ground-truth-verb decode of the imSitu gt-value metrics.

        Inference only, in train mode too: no autograd node is built and no dropout is applied.  Honours
        `self.precision`, and makes no host synchronisation (it can be captured in a CUDA graph).  Returns
        `Situations`."""
        fn = _as_feat(feat_nouns, self.D)
        dev = fn.device
        eng = self._engine_for(dev)
        B = fn.shape[0]
        if verbs is not None:
            verbs = verbs.to(device=dev, dtype=torch.int64).contiguous()
            if verbs.dim() != 2 or verbs.shape[0] != B:
                raise _lib.SrgError("verbs must be [B, k] = [%d, k], got %s" % (B, tuple(verbs.shape)))
            k = verbs.shape[1]
        if not 1 <= k <= min(MAX_TOPK, eng.V):
            raise _lib.SrgError("k=%d must be in [1, %d]" % (k, min(MAX_TOPK, eng.V)))
        prec = _prec_code(self.precision)
        eng.ensure_packed(self, prec)
        stream = eng.stream()
        verb_logp = None
        if verbs is None:
            fv = _as_feat(feat_verbs, self.D)
            if fv.shape[0] != B:
                raise _lib.SrgError("feat_verbs has %d rows, feat_nouns %d" % (fv.shape[0], B))
            logits = torch.empty(B, eng.Vpad, dtype=torch.float32, device=dev)
            ws = eng.workspace(SRG_MODE_VERB, B, prec, False)
            _lib.check(eng.lib.srg_verb_forward(eng.h, _lib.ptr(fv), B, None, 0.0, None, 0, _lib.ptr(logits), eng.Vpad,
                                                prec, 0, _lib.ptr(ws), ws.numel(), stream))
            verbs = torch.empty(B, k, dtype=torch.int64, device=dev)
            verb_logp = torch.empty(B, k, dtype=torch.float32, device=dev)
            _lib.check(eng.lib.srg_topk_logsoftmax(_lib.ptr(logits), eng.Vpad, B, eng.V, k, _lib.ptr(verbs),
                                                   _lib.ptr(verb_logp), stream))
        labels = torch.empty(B, k, eng.R, dtype=torch.int64, device=dev)
        label_logp = torch.empty(B, k, eng.R, dtype=torch.float32, device=dev)
        score = torch.empty(B, k, dtype=torch.float32, device=dev)
        ws = eng.workspace(SRG_MODE_NOUN, B, prec, False, k=k)
        _lib.check(eng.lib.srg_situation_nouns(eng.h, _lib.ptr(fn), _lib.ptr(verbs), B, k, _lib.ptr(self.role_emb.weight),
                                               _lib.ptr(self.verb_emb.weight), _lib.ptr(verb_logp), _lib.ptr(labels),
                                               _lib.ptr(label_logp), _lib.ptr(score), prec, _lib.ptr(ws), ws.numel(),
                                               stream))
        return Situations(verbs, verb_logp, labels, label_logp, score)

    @torch.no_grad()
    def nbest_situations_from_features(self, feat_verbs, feat_nouns, n=5, verb_beam=None, verbs=None):
        """The n highest-scoring situations of each image from the backbone features ([B, D] each), and whether the
        list is certified to be the n-best over all verbs.  Returns `(Situations, exact)`, `exact` bool [B].

        A situation is one of the kv = verb_beam (default n, at most 15) best verbs plus one label per role of that
        verb; its score is verb_logp + l_0 + l_1 + ... summed in fp32 in slot order, l_r the label's log-softmax over
        the labels.  Order: score descending, then the better-ranked verb, then the per-slot label ranks compared
        lexicographically from slot 0.  The 1-best entry is bit-identical to the best-scoring candidate of
        `situations_from_features(k=kv)`.  Situations whose scores lie within one fp32 rounding of each other may come
        out in either order.  exact[b]: score[b, n-1] >= the log-prob of the (kv+1)-th verb, so no situation of a verb
        outside the beam can enter the list (every label log-prob is <= 0).
        verbs ([B, kv'] int64, optional): decode these candidate verbs instead (feat_verbs is then not used and may be
        None; verb_logp is None, the score is the label term only and exact is all True) -- e.g. `verbs=v[:, None]`
        for the n best label assignments of verb v.

        Same rules as `situations_from_features`: no autograd node, no dropout, no host synchronisation (it can be
        captured in a CUDA graph), honours `self.precision`."""
        fn = _as_feat(feat_nouns, self.D)
        dev = fn.device
        eng = self._engine_for(dev)
        B = fn.shape[0]
        if not 1 <= n <= min(MAX_TOPK, eng.L):
            raise _lib.SrgError("n=%d must be in [1, %d]" % (n, min(MAX_TOPK, eng.L)))
        if verbs is not None:
            verbs = verbs.to(device=dev, dtype=torch.int64).contiguous()
            if verbs.dim() != 2 or verbs.shape[0] != B:
                raise _lib.SrgError("verbs must be [B, kv] = [%d, kv], got %s" % (B, tuple(verbs.shape)))
            kv = verbs.shape[1]
            if not 1 <= kv <= min(MAX_TOPK, eng.V):
                raise _lib.SrgError("verbs has %d columns, must be in [1, %d]" % (kv, min(MAX_TOPK, eng.V)))
        else:
            kv = n if verb_beam is None else verb_beam
            if not 1 <= kv <= min(MAX_VERB_BEAM, eng.V):
                raise _lib.SrgError("verb_beam=%d must be in [1, %d]" % (kv, min(MAX_VERB_BEAM, eng.V)))
        prec = _prec_code(self.precision)
        eng.ensure_packed(self, prec)
        stream = eng.stream()
        verb_logp = verb_bound = None
        if verbs is None:
            fv = _as_feat(feat_verbs, self.D)
            if fv.shape[0] != B:
                raise _lib.SrgError("feat_verbs has %d rows, feat_nouns %d" % (fv.shape[0], B))
            logits = torch.empty(B, eng.Vpad, dtype=torch.float32, device=dev)
            ws = eng.workspace(SRG_MODE_VERB, B, prec, False)
            _lib.check(eng.lib.srg_verb_forward(eng.h, _lib.ptr(fv), B, None, 0.0, None, 0, _lib.ptr(logits), eng.Vpad,
                                                prec, 0, _lib.ptr(ws), ws.numel(), stream))
            kt = min(kv + 1, eng.V)              # kt = kv: every verb is in the beam, nothing to bound
            top = torch.empty(B, kt, dtype=torch.int64, device=dev)
            top_logp = torch.empty(B, kt, dtype=torch.float32, device=dev)
            _lib.check(eng.lib.srg_topk_logsoftmax(_lib.ptr(logits), eng.Vpad, B, eng.V, kt, _lib.ptr(top),
                                                   _lib.ptr(top_logp), stream))
            verbs, verb_logp = top[:, :kv].contiguous(), top_logp[:, :kv].contiguous()
            if kt > kv:
                verb_bound = top_logp[:, kv].contiguous()
        out_verbs = torch.empty(B, n, dtype=torch.int64, device=dev)
        out_verb_logp = None if verb_logp is None else torch.empty(B, n, dtype=torch.float32, device=dev)
        labels = torch.empty(B, n, eng.R, dtype=torch.int64, device=dev)
        label_logp = torch.empty(B, n, eng.R, dtype=torch.float32, device=dev)
        score = torch.empty(B, n, dtype=torch.float32, device=dev)
        exact = torch.empty(B, dtype=torch.bool, device=dev)             # the kernel stores one byte 0 / 1 per image
        ws = eng.workspace(SRG_MODE_NOUN, B, prec, False, k=kv, nbest=n)
        _lib.check(eng.lib.srg_situation_nbest(eng.h, _lib.ptr(fn), _lib.ptr(verbs), B, kv, _lib.ptr(self.role_emb.weight),
                                               _lib.ptr(self.verb_emb.weight), _lib.ptr(verb_logp),
                                               _lib.ptr(verb_bound), n, _lib.ptr(out_verbs), _lib.ptr(out_verb_logp),
                                               _lib.ptr(labels), _lib.ptr(label_logp), _lib.ptr(score),
                                               _lib.ptr(exact), prec, _lib.ptr(ws), ws.numel(), stream))
        return Situations(out_verbs, out_verb_logp, labels, label_logp, score), exact

    @torch.no_grad()
    def predict_situations(self, img, k=5, img_nouns=None):
        """`situations_from_features` from images, through the two backbones (same rules: no autograd, no
        dropout, no host synchronisation)."""
        fv, fn = self.extract_features(img, img_nouns)
        return self.situations_from_features(fv, fn, k=k)

    # ---- GGSNN.forward drop-in ------------------------------------------------------------------
    def _ggsnn_forward(self, hidden_state, mask=None, verb=False):
        if not hidden_state.is_cuda:
            raise _lib.SrgError("the GGNN stage has no CPU path: hidden_state must be a CUDA tensor")
        eng = self._engine_for(hidden_state.device)
        prec = _prec_code(self.precision)
        mask = None if verb else mask
        params = self._ggnn_params()
        need_grad = torch.is_grad_enabled() and any(
            t is not None and t.requires_grad for t in [hidden_state, mask] + params)
        if not verb and mask is None:
            raise _lib.SrgError("GGSNN.forward on the role graph (verb=False) needs a mask")
        if need_grad:
            if prec != SRG_PREC_BF16:
                raise _lib.SrgError("precision='fp32' is a forward-only parity mode; use torch.no_grad() or "
                                    "precision='bf16'")
            return _GGSNNStage.apply(self, hidden_state, mask, *params)
        eng.ensure_packed(self, prec)
        h, mode, B, mk = _ggsnn_inputs(eng, hidden_state, mask, verb)
        ws = eng.workspace(mode, B, prec, False)
        _lib.check(eng.lib.srg_ggnn_forward(eng.h, mode, _lib.ptr(h), _lib.ptr(mk), B, prec, 0, _lib.ptr(ws),
                                            ws.numel(), eng.stream()))
        return h

    def check_verbs(self, device=None):
        """Raise SrgError if any predict_nouns / forward call since the last check saw a verb id outside
        [0, num_verbs) (the kernels clamp such ids to 0 instead of faulting; the reference raises an IndexError).
        Synchronises the stream: call it when debugging data, not in the training loop."""
        for key, eng in self._engines.items():
            if device is None or torch.device(device).index in (None, key[1]):
                _lib.check(eng.lib.srg_check_verbs(eng.h, eng.stream()))

    def gather_mask(self, verbs):
        """CUDA replacement of encoder.get_role_ids_batch + get_adj_matrix_noself (imsitu_encoder.py:172-180,209-229)."""
        if not verbs.is_cuda:
            raise _lib.SrgError("gather_mask needs a CUDA tensor of verb ids")
        eng = self._engine_for(verbs.device)
        v = verbs.detach().to(torch.int64).contiguous()
        B = v.shape[0]
        R = eng.R
        role_idx = torch.empty(B, R, dtype=torch.int64, device=v.device)
        mask = torch.empty(B, R, R, dtype=torch.float32, device=v.device)
        bad = torch.zeros(1, dtype=torch.int32, device=v.device)
        _lib.check(eng.lib.srg_gather_mask(eng.h, _lib.ptr(v), B, _lib.ptr(role_idx), _lib.ptr(mask), _lib.ptr(bad),
                                           eng.stream()))
        return role_idx, mask, bad
