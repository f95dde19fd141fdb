"""Cross-epoch cache of the frozen backbones' features (SURVEY.md section 8f, N3).

Both ResNet-152 backbones of the reference are frozen (`requires_grad = False`, model.py:17-18; sr.py:488-503 re-freezes
them after a resume) and, in evaluation, run in eval mode on a deterministic transform (`dev_transform`:
Resize -> CenterCrop -> ToTensor -> Normalize, imsitu_encoder.py:27-36).  The 2 x 2048 features of a dev / test image are
therefore the same in every epoch, while the reference recomputes three ResNet-152 passes per image every time
(model.py:116,159,175-178) -- 92 % of an end-to-end eval step on a B200.  The cache stores them once, on the GPU
(25 200 dev images x 2 x 2048 fp32 = 413 MB), and later epochs feed `FCGGNN.forward_features` directly.

The cache is only valid for frozen backbones: `sr.py --finetune_backbone` (or any caller that trains a backbone) must
not use it, since the features then change at every optimizer step.

Training features are NOT cached by the launcher: the reference trains with random crops / flips and with the backbones'
BatchNorm layers in training mode (model.train(), sr.py:24), so those features legitimately change every epoch.
"""
import torch


class FeatureCache:
    def __init__(self, capacity, D, device, dtype=torch.float32):
        self.D = D
        self.index = {}                      # image name -> row
        self.feat_v = torch.empty(capacity, D, dtype=dtype, device=device)
        self.feat_n = torch.empty(capacity, D, dtype=dtype, device=device)
        self.hits = 0
        self.misses = 0

    def __len__(self):
        return len(self.index)

    def has(self, names):
        return all(n in self.index for n in names)

    def lookup(self, names):
        """(feat_verbs, feat_nouns) fp32 [B, D] for `names`, or None unless every one of them is cached."""
        try:
            rows = [self.index[n] for n in names]
        except KeyError:
            self.misses += len(names)
            return None
        self.hits += len(names)
        idx = torch.tensor(rows, dtype=torch.int64, device=self.feat_v.device)
        return self.feat_v.index_select(0, idx).float(), self.feat_n.index_select(0, idx).float()

    def store(self, names, feat_v, feat_n):
        rows = []
        for n in names:
            r = self.index.get(n)
            if r is None:
                r = len(self.index)
                if r >= self.feat_v.shape[0]:
                    raise ValueError("FeatureCache capacity %d exceeded" % self.feat_v.shape[0])
                self.index[n] = r
            rows.append(r)
        idx = torch.tensor(rows, dtype=torch.int64, device=self.feat_v.device)
        self.feat_v.index_copy_(0, idx, feat_v.detach().to(self.feat_v.dtype))
        self.feat_n.index_copy_(0, idx, feat_n.detach().to(self.feat_n.dtype))

    def features(self, model, names, img):
        """Cached features of the batch, computing (and storing) them with the model's backbones on a miss.  `img` may
        be None / empty when the caller knows the batch is cached (`has`)."""
        got = self.lookup(names)
        if got is not None:
            return got
        with torch.no_grad():
            fv, fn = model.extract_features(img)
        self.store(names, fv, fn)
        return fv, fn
