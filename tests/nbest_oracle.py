"""Test oracle of the n-best situation decode (FCGGNN.nbest_situations_from_features, srg_situation_nbest).  Test
infrastructure only.

A candidate is (verb_logp or None, lp) with lp [nr, m]: the label log-probs of its nr real role slots in rank order
(rank = position in a stable descending sort of the slot's labels, ties to the lower label).  A situation is
(candidate j, ranks), its score verb_logp + lp[0, rank_0] + lp[1, rank_1] + ..., added one term at a time in slot
order in lp's dtype (fp32 rounds exactly as the kernel does; fp64 for the fp64 parity checks).  Order: score
descending, then lower j, then the ranks compared lexicographically from slot 0.
"""
import heapq
import itertools

import numpy as np
import torch


def rank_lists(logp, m=None):
    """logp [..., L] (torch) -> (label ids [..., m], log-probs [..., m]) by a stable descending sort."""
    order = torch.sort(logp, dim=-1, descending=True, stable=True).indices
    if m is not None:
        order = order[..., :m]
    return order, logp.gather(-1, order)


def _score(vlp, lp, ranks):
    s = lp.dtype.type(0) if vlp is None else lp.dtype.type(vlp)
    for r, k in enumerate(ranks):
        s = lp.dtype.type(s + lp[r, k])
    return s


def _key(entry):
    s, j, ranks = entry
    return (-float(s), j, ranks)


def nbest_enumerate(cands, n):
    """Every label assignment of every candidate, sorted by the order; the first n (fewer when fewer exist)."""
    out = []
    for j, (vlp, lp) in enumerate(cands):
        lp = np.asarray(lp)
        for ranks in itertools.product(*[range(lp.shape[1])] * lp.shape[0]):
            out.append((_score(vlp, lp, ranks), j, ranks))
    return sorted(out, key=_key)[:n]


def nbest_best_first(cands, n):
    """The same list as nbest_enumerate, without enumerating: per candidate, pop the best of a frontier that starts at
    the all-zero ranks and grows by raising one slot's rank.  Raising a rank never raises the score (fp rounding is
    monotone) and makes the ranks lexicographically larger, so every situation ranks after the ones it grew from and
    the pops come out in order."""
    out = []
    for j, (vlp, lp) in enumerate(cands):
        lp = np.asarray(lp)
        nr, m = lp.shape
        start = (0,) * nr
        heap = [_key((_score(vlp, lp, start), j, start)) + (_score(vlp, lp, start),)]
        seen = {start}
        for _ in range(n):
            if not heap:
                break
            _, _, ranks, s = heapq.heappop(heap)
            out.append((s, j, ranks))
            for r in range(nr):
                if ranks[r] + 1 < m:
                    nxt = ranks[:r] + (ranks[r] + 1,) + ranks[r + 1:]
                    if nxt not in seen:
                        seen.add(nxt)
                        sn = _score(vlp, lp, nxt)
                        heapq.heappush(heap, _key((sn, j, nxt)) + (sn,))
    return sorted(out, key=_key)[:n]


def certified(beam_list, n, verb_bound):
    """exact: the beam's n-th score is at least the log-prob of the best verb outside the beam."""
    return verb_bound is None or (len(beam_list) == n and float(beam_list[-1][0]) >= float(verb_bound))
