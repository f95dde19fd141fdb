"""CPU checks of the top-k situation decode's host side: the standard imSitu metrics of `situations.SituationScorer`
against a plain loop over their definitions, and the decode oracle (tests/situations_oracle.py) against a per-image loop of
predict_verb / predict_nouns."""
import pytest
import torch

import situation_recognition_b200 as S
from oracle import ggnn_oracle as O
from tests.situations_oracle import situations
from situation_recognition_b200.model import Situations
from situation_recognition_b200.situations import SituationScorer
from situation_recognition_b200.synthetic import make_train_json


@pytest.fixture(scope="module")
def enc():
    return S.imsitu_encoder(make_train_json(seed=0, images_per_verb=1), verbose=False)


def loop_metrics(enc, verbs, labels, gt_verb, gt_nouns, gt_labels, ks):
    """The definitions, one image and one candidate at a time."""
    L = enc.get_num_labels()
    tot = {}
    for b in range(len(gt_verb)):
        gv = int(gt_verb[b])
        n = enc.get_role_count(gv)

        def correct(lab):
            ok = [int(lab[r]) in [int(x) for x in gt_nouns[b, :, r] if int(x) != L] for r in range(n)]
            return sum(ok) / max(n, 1), all(ok)

        for k in ks:
            vals = {"verb@%d" % k: 0.0, "value@%d" % k: 0.0, "value-all@%d" % k: 0.0}
            for j in range(k):
                if int(verbs[b, j]) == gv:
                    v, a = correct(labels[b, j])
                    vals = {"verb@%d" % k: 1.0, "value@%d" % k: v, "value-all@%d" % k: float(a)}
                    break
            for key, x in vals.items():
                tot[key] = tot.get(key, 0.0) + x
        v, a = correct(gt_labels[b, 0])
        tot["gt-value"] = tot.get("gt-value", 0.0) + v
        tot["gt-value-all"] = tot.get("gt-value-all", 0.0) + float(a)
    out = {key: x / len(gt_verb) for key, x in tot.items()}
    out["mean"] = sum(out.values()) / len(out)
    return out


def random_batch(enc, B, K, seed):
    """Candidates with the gt verb at every position (and absent), labels drawn from a small pool so that they often
    tie with an annotation, pad annotations (= num_labels) beyond each gt verb's roles and in some real roles."""
    g = torch.Generator().manual_seed(seed)
    V, R, L = enc.get_num_verbs(), enc.get_max_role_count(), enc.get_num_labels()
    gt_verb = torch.randint(0, V, (B,), generator=g)
    verbs = torch.stack([torch.randperm(V, generator=g)[:K] for _ in range(B)])
    pos = torch.randint(0, K + 1, (B,), generator=g)            # K = gt verb not among the candidates
    for b in range(B):
        verbs[b][verbs[b] == gt_verb[b]] = (gt_verb[b] + 1) % V
        if pos[b] < K:
            verbs[b, pos[b]] = gt_verb[b]
    gt_nouns = torch.randint(0, 4, (B, 3, R), generator=g)
    gt_nouns[torch.rand(B, 3, R, generator=g) < 0.2] = L       # some annotators left a real role empty
    counts = torch.tensor([enc.get_role_count(int(v)) for v in gt_verb])
    gt_nouns[(torch.arange(R)[None, None, :] >= counts[:, None, None]).expand(B, 3, R)] = L
    labels = torch.randint(0, 4, (B, K, R), generator=g)
    vc = torch.tensor([[enc.get_role_count(int(v)) for v in row] for row in verbs])
    labels[torch.arange(R)[None, None, :] >= vc[:, :, None]] = -1
    gt_labels = torch.randint(0, 4, (B, 1, R), generator=g)
    gt_labels[torch.arange(R)[None, None, :] >= counts[:, None, None]] = -1
    return verbs, labels, gt_verb, gt_nouns, gt_labels


def sit(verbs, labels):
    z = torch.zeros(labels.shape)
    return Situations(verbs, None, labels, z, z.sum(-1))


@pytest.mark.parametrize("ks,K", [((1, 5), 5), ((1, 3), 7), ((1,), 1)])
def test_scorer_matches_definition_loop(enc, ks, K):
    scorer = SituationScorer(enc, ks)
    batches = [random_batch(enc, B, K, seed) for seed, B in ((0, 64), (1, 37), (2, 1))]
    for verbs, labels, gt_verb, gt_nouns, gt_labels in batches:
        scorer.add_point(sit(verbs, labels), gt_verb, gt_nouns, sit(gt_verb[:, None], gt_labels))
    got = scorer.get_average_results()
    cat = [torch.cat(x) for x in zip(*batches)]
    ref = loop_metrics(enc, *cat, ks=scorer.ks)
    assert set(got) == set(ref)
    for key in ref:
        assert got[key] == pytest.approx(ref[key], abs=1e-12), key
    # the positions cover every rank of the candidate list, and misses
    assert 0.0 < got["verb@%d" % ks[0]] < 1.0


def test_scorer_rejects_too_few_candidates(enc):
    verbs, labels, gt_verb, gt_nouns, gt_labels = random_batch(enc, 4, 3, 0)
    with pytest.raises(ValueError):
        SituationScorer(enc, (1, 5)).add_point(sit(verbs, labels), gt_verb, gt_nouns, sit(gt_verb[:, None], gt_labels))


@pytest.mark.parametrize("given", [False, True])
def test_oracle_situations_match_per_image_loop(enc, given):
    D, B, k = 16, 6, 5
    params = O.init_params(enc.get_num_verbs(), enc.get_num_roles(), enc.get_num_labels(), D, seed=3,
                           dtype=torch.float64)
    g = torch.Generator().manual_seed(4)
    fv, fn = torch.rand(B, D, generator=g, dtype=torch.float64), torch.rand(B, D, generator=g, dtype=torch.float64)
    t, c = O.build_tables(enc.roles_per_verb, enc.verb_list, enc.role_list)
    given_verbs = torch.randint(0, enc.get_num_verbs(), (B, 2), generator=g) if given else None
    verbs, verb_logp, labels, label_logp, score = situations(params, fv, fn, k, t, c, verbs=given_verbs)
    for b in range(B):
        if given:
            cand, vlp = given_verbs[b], None
            assert verb_logp is None
        else:
            pv = O.predict_verb(params, fv[b:b + 1])[0]
            lp = torch.log_softmax(pv, 0)
            cand = []
            rest = pv.clone()
            for _ in range(k):                       # repeated argmax = stable descending sort
                i = int(torch.argmax(rest))
                cand.append(i)
                rest[i] = -float("inf")
            assert verbs[b].tolist() == cand
            vlp = lp[cand]
            assert torch.allclose(verb_logp[b], vlp, atol=1e-12)
        for j, v in enumerate(cand):
            nl = O.predict_nouns(params, fn[b:b + 1], torch.tensor([int(v)]), t, c)[0]       # [R, L]
            n = int(c[int(v)])
            assert labels[b, j, :n].tolist() == torch.argmax(nl, -1)[:n].tolist()
            assert (labels[b, j, n:] == -1).all() and (label_logp[b, j, n:] == 0).all()
            lp = torch.log_softmax(nl, -1).max(-1).values[:n]
            assert torch.allclose(label_logp[b, j, :n], lp, atol=1e-12)
            expect = lp.sum() + (vlp[j] if vlp is not None else 0)
            assert abs(float(score[b, j]) - float(expect)) < 1e-10


@pytest.mark.parametrize("argv", [["--evaluate_dev", "--topk_situations", "1"],
                                  ["--evaluate_test", "--topk_situations", "1"],
                                  ["--test_img", "x.jpg", "--topk_situations", "17"],
                                  ["--topk_situations", "-1"]])
def test_launcher_rejects_topk_situations_out_of_range(argv):
    """The evaluation block reports top-1 and top-K and the mean of those 8 numbers, so K = 1 is refused there; the
    decode takes at most 16 candidates.  Refused while parsing, before anything touches a GPU."""
    from situation_recognition_b200 import sr
    with pytest.raises(SystemExit) as e:
        sr.main(argv)
    assert e.value.code == 2
