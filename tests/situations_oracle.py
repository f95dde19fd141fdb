"""Test oracle of the top-k situation decode (FCGGNN.situations_from_features), built only from the CPU oracle's
predict_verb / predict_nouns (oracle/ggnn_oracle.py) plus an fp64 log_softmax and a stable sort.  Test infrastructure
only."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import ggnn_oracle as O


def situations(params, feat_verbs, feat_nouns, k, verb2roles, role_count, verbs=None):
    """Top-k situation decode (FCGGNN.situations_from_features) from predict_verb / predict_nouns, without dropout.
    Candidates: the k largest verb logits by a stable descending sort (ties to the lower id), or `verbs` [B, k'] when
    given (verb_logp is then None).  Per candidate the top-1 label of every role slot (stable sort) with its fp64
    log_softmax over the labels; pad slots -1 / 0.  score = verb_logp (or 0) + sum of the real slots' label log-probs.
    Returns (verbs, verb_logp, labels, label_logp, score); log-probs and scores in fp64."""
    B, R = feat_nouns.shape[0], verb2roles.shape[1]
    verb_logp = None
    if verbs is None:
        pv = O.predict_verb(params, feat_verbs)
        verbs = torch.sort(pv, dim=1, descending=True, stable=True).indices[:, :k]
        verb_logp = F.log_softmax(pv.double(), dim=1).gather(1, verbs)
    k = verbs.shape[1]
    counts = torch.as_tensor(np.asarray(role_count), dtype=torch.int64)
    labels = torch.full((B, k, R), -1, dtype=torch.int64)
    label_logp = torch.zeros(B, k, R, dtype=torch.float64)
    for j in range(k):
        nl = O.predict_nouns(params, feat_nouns, verbs[:, j], verb2roles, role_count, keep=None)      # [B, R, L]
        top = torch.sort(nl, dim=-1, descending=True, stable=True).indices[..., :1]
        lp = F.log_softmax(nl.double(), dim=-1).gather(-1, top)[..., 0]
        real = torch.arange(R)[None, :] < counts[verbs[:, j]][:, None]
        labels[:, j] = torch.where(real, top[..., 0], torch.full_like(top[..., 0], -1))
        label_logp[:, j] = torch.where(real, lp, torch.zeros_like(lp))
    score = label_logp.sum(-1) + (verb_logp if verb_logp is not None else 0)
    return verbs, verb_logp, labels, label_logp, score
