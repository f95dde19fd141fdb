"""Standard imSitu top-k situation metrics on the decode of `FCGGNN.situations_from_features`.

A situation is a verb plus one label per role of that verb.  These are the definitions the imSitu literature reports
(top-1 / top-5 verb, value, value-all, gt-value, gt-value-all), not the reference scorer's (`imsitu_scorer.py`, whose
"top-5" ranks the nouns of each role under the argmax verb).  Per image, with the gt verb's n roles and the three
annotations of each role:
  * verb@k      1 if the gt verb is among the first k candidate verbs;
  * value@k     if the gt verb is candidate j < k: the mean over its n roles of [predicted label is one of the role's
                three annotations]; otherwise 0;
  * value-all@k 1 if the gt verb is candidate j < k and all n roles of that candidate are correct, else 0;
  * gt-value, gt-value-all  value / value-all of the decode conditioned on the gt verb (`verbs = gt_verb[:, None]`);
  * mean        the average of all of the above: 3 * len(ks) + 2 numbers, i.e. the 8 of the literature for ks = (1, 5)
                (ks = (1,) gives a 5-number mean that is not comparable with it).
Everything stays on the device; the averages cost one device-to-host copy when they are read.
"""
import torch


class SituationScorer:
    def __init__(self, encoder, ks=(1, 5)):
        self.encoder = encoder
        self.ks = tuple(sorted(set(int(k) for k in ks)))
        if not self.ks or self.ks[0] < 1:
            raise ValueError("ks must be positive, got %s" % (ks,))
        self.keys = [m + "@%d" % k for k in self.ks for m in ("verb", "value", "value-all")] + ["gt-value",
                                                                                                 "gt-value-all"]
        self._sums = None            # device fp64 [len(keys)]; sr._merge_scorer all-reduces _sums and _count
        self._count = 0
        self._role_count = None

    def _counts_for(self, verbs):
        if self._role_count is None or self._role_count.device != verbs.device:
            n = self.encoder.get_num_verbs()
            self._role_count = torch.tensor([self.encoder.get_role_count(v) for v in range(n)], dtype=torch.int64,
                                            device=verbs.device)
        return self._role_count[verbs]

    @staticmethod
    def _correct(labels, gt_nouns, valid):
        """labels [B,K,R], gt_nouns [B,3,R], valid [B,R] -> (value [B,K], value_all [B,K]) of each candidate's labels
        against the gt verb's roles."""
        hit = (labels[:, :, :, None] == gt_nouns.transpose(1, 2)[:, None, :, :]).any(-1) & valid[:, None, :]
        n = valid.sum(1).clamp_min(1)[:, None]
        return hit.sum(-1).to(torch.float64) / n, hit.sum(-1) == valid.sum(1)[:, None]

    @torch.no_grad()
    def add_point(self, situations, gt_verb, gt_nouns, gt_situations):
        """situations: the top-k decode (`Situations`, at least max(ks) candidates); gt_verb [B]; gt_nouns [B,3,R]
        (pad = num_labels); gt_situations: the decode with verbs = gt_verb[:, None]."""
        verbs, labels = situations.verbs, situations.labels
        B, K, R = labels.shape
        if B == 0:
            return
        if K < self.ks[-1]:
            raise ValueError("%d candidates per image, top-%d needs at least that many" % (K, self.ks[-1]))
        dev = labels.device
        gt_verb = gt_verb.to(dev).long()
        gt_nouns = gt_nouns.to(dev).long()
        valid = torch.arange(R, device=dev)[None, :] < self._counts_for(gt_verb)[:, None]            # [B,R]
        value, value_all = self._correct(labels, gt_nouns, valid)
        hit = verbs == gt_verb[:, None]                                                             # [B,K]
        first = hit & (hit.cumsum(1) == 1)                       # the gt verb's candidate (first one, were it repeated)
        cols = []
        for k in self.ks:
            f = first[:, :k]
            cols += [f.any(1).to(torch.float64), (value[:, :k] * f).sum(1), (value_all[:, :k] & f).any(1).to(torch.float64)]
        g_value, g_all = self._correct(gt_situations.labels[:, :1], gt_nouns, valid)
        cols += [g_value[:, 0], g_all[:, 0].to(torch.float64)]
        s = torch.stack(cols, 1).sum(0)
        self._sums = s if self._sums is None else self._sums + s.to(self._sums.device)
        self._count += B

    def get_average_results(self):
        """{key: fraction} for every key plus "mean" (the average of those 3 * len(ks) + 2 numbers); one device-to-host
        copy."""
        sums = self._sums.cpu().tolist() if self._sums is not None else [0.0] * len(self.keys)
        out = {key: s / self._count for key, s in zip(self.keys, sums)}     # ZeroDivisionError on an empty scorer
        out["mean"] = sum(out.values()) / len(self.keys)
        return out
