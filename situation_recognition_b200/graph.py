"""CUDA-graph capture of one GGNN training step.

A step launches ~130 kernels of this library (67 tensor-core GEMMs, the HBM-bound kernels, clip + Adamax) plus ~30 small
torch kernels and the NCCL collectives.  At the full 6144-image batch the host queues them faster than the GPU runs
them; on a 768-image shard (8 GPUs) queueing a step takes about as long as executing it.  The whole step -- weight
packing, the three forward paths (including the device-side argmax of the predicted verb, the device-resident row counts
of the compact role-node layout and the Philox dropout seed), the losses, the backward pass, the NCCL collectives, clip
and the optimizer -- has no host synchronisation, so it is captured once into a CUDA graph with static input buffers
and replayed.
"""
import torch

from . import _lib


class GraphedTrainStep:
    """step(feat_verbs, feat_nouns, gt_verb, gt_nouns) -> fp32[3] (verb_loss, nouns_loss, gt_nouns_loss).

    Mirrors the body of the reference's training loop (sr.py:63-83) without AMP:
        zero grads; model(img, verb); verb_loss, nouns_loss, gt_nouns_loss; (verb_loss + nouns_loss).backward();
        [all-reduce]; clip_grad_norm_(params, clip); optimizer.step()
    `optimizer` must be capturable: parallel.FlatAdamax (fused clip + Adamax kernel) or
    torch.optim.Adamax(..., capturable=True).  Inputs may live on the host
    (pinned) or on the device; they are copied into the graph's static buffers before each replay.
    verb_loss_kwargs / nouns_loss_kwargs: the training objective's `weight`, `label_smoothing` and `reduction`
    ("mean" or "sum") of verb_loss and of both nouns_loss calls.  The captured step reads the weight tensors in place.
    """

    def __init__(self, model, optimizer, flat, batch, clip=1.0, warmup=3, verb_loss_kwargs=None,
                 nouns_loss_kwargs=None):
        self.model, self.opt, self.flat, self.clip = model, optimizer, flat, clip
        self.verb_kw, self.nouns_kw = dict(verb_loss_kwargs or {}), dict(nouns_loss_kwargs or {})
        for kw in (self.verb_kw, self.nouns_kw):
            if kw.get("reduction", "mean") not in ("mean", "sum"):
                raise ValueError("GraphedTrainStep back-propagates a scalar loss: reduction must be 'mean' or 'sum'")
        dev = next(model.parameters()).device
        enc = model.encoder
        R = enc.get_max_role_count()
        self.static_in = (torch.zeros(batch, model.D, device=dev), torch.zeros(batch, model.D, device=dev),
                          torch.zeros(batch, dtype=torch.int64, device=dev),
                          torch.full((batch, 3, R), enc.get_num_labels(), dtype=torch.int64, device=dev))
        self.params = [p for p in model.parameters() if p.requires_grad]
        self.graph = None
        self.losses = None
        self.launches = 0
        self._warmup = warmup

    def _body(self):
        a, b, v, n = self.static_in
        m = self.model
        self.flat.zero()
        pred_verb, pred_nouns, gt_pred_nouns = m(a, v, img_nouns=b)
        vl = m.verb_loss(pred_verb, v, **self.verb_kw)
        nl = m.nouns_loss(pred_nouns, n, **self.nouns_kw)
        gl = m.nouns_loss(gt_pred_nouns, n, **self.nouns_kw)
        (vl + nl).backward()
        if getattr(self.opt, "world", 1) <= 1:      # a sharded FlatAdamax reduce-scatters the gradient itself
            self.flat.all_reduce()
        if not getattr(self.opt, "fused_clip", False):
            torch.nn.utils.clip_grad_norm_(self.params, self.clip)
        self.opt.step()                         # FlatAdamax clips inside its fused kernel
        return torch.stack([vl.detach(), nl.detach(), gl.detach()])

    def capture(self, example):
        for dst, src in zip(self.static_in, example):
            dst.copy_(src)
        lib = _lib.load()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(self._warmup):
                self._body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for eng in self.model._engines.values():
            eng._packed_key = None              # make the weight packing part of the captured step
        self.graph = torch.cuda.CUDAGraph()
        n0 = lib.srg_launch_count()
        with torch.cuda.graph(self.graph):
            self.losses = self._body()
        self.launches = lib.srg_launch_count() - n0
        for eng in self.model._engines.values():
            eng._packed_key = None              # the graph repacks on every replay; eager calls must repack too
        return self

    def __call__(self, feat_verbs, feat_nouns, gt_verb, gt_nouns):
        if self.graph is None:
            self.capture((feat_verbs, feat_nouns, gt_verb, gt_nouns))
        else:
            for dst, src in zip(self.static_in, (feat_verbs, feat_nouns, gt_verb, gt_nouns)):
                if src is not dst:
                    dst.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.losses
