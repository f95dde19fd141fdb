"""-m gpu: the stage at hidden sizes, role counts and vocabularies other than the rest of the suite's two (D = 256 / R = 4
and D = 2048 / R = 6 / 504 verbs / 2001 labels), against the fp64 oracle.  Each row of GEOMETRIES reaches shapes that
only it runs:

  D = 512,  R = 8, 37 / 23 / 257      R = kMaxR (register arrays of the aggregation, node-init and row-map kernels), slot 7
                                      of the n-best rank packing (bits 0..3), a padded label tile holding one column
  D = 768,  R = 3, 504 / 190 / 2001   an odd number of 256-column N tiles in the N = D GEMMs at cta_group 2
  D = 1280, R = 6, 129 / 40 / 511     D / 8 = 160 column groups: partial second passes in the D/8-sized kernels
  D = 256,  R = 1, 11 / 5 / 13        no neighbours (all-zero adjacency), 0-role verbs, n-best with n = 13 < 16
  D = 1024, R = 5, 300 / 90 / 4200    Lpad / 128 = 34 > 32 softmax-statistics tiles: the fused training step takes the
                                      loss kernels' three-pass route

Every vocabulary has verbs of each role count 0..R (tests/geometry.py).  Each geometry runs on both row layouts (compact
rows and one row per slot) and both cta_groups, at B = 1 and at the smallest batch whose compact rows straddle a
256-row tile boundary inside one image (geometry.crossing_verbs; at R = 1 the row count passes 256).  Bounds are the
suite's (tests/test_gpu_parity.py): fp32 mode 1e-4 of max|ref| with the same argmax on >= 99.9 % of the rows, bf16
logits 2e-2, losses 2e-3 relative, every gradient 3e-2.  The oracle runs in fp64, on the GPU (the top-k decode's on
the CPU).  Each case prints a `PARITY {json}` line with its errors.  The whole module (115 cases) takes about 15 s on
one B200 (1000 W power limit)."""
import functools
import json

import numpy as np
import pytest
import torch

import situation_recognition_b200 as S
from oracle import ggnn_oracle as O
from situation_recognition_b200 import _lib
from tests import geometry as GE
from tests import regimes as G
from tests.situations_oracle import situations as oracle_situations
from tests.test_nbest_gpu import beam, check_self_consistent, compare, oracle_lists, slot_lists

pytestmark = pytest.mark.gpu

FP32_TOL, LOGIT_TOL, LOSS_TOL, GRAD_TOL, LAYOUT_TOL = 1e-4, 2e-2, 2e-3, 3e-2, 2e-3
GEOMETRIES = {"D512_R8": (512, 8, 37, 23, 257), "D768_R3": (768, 3, 504, 190, 2001),
              "D1280_R6": (1280, 6, 129, 40, 511), "D256_R1": (256, 1, 11, 5, 13),
              "D1024_R5": (1024, 5, 300, 90, 4200)}
LAYOUTS = {"compact": True, "per_slot": False}
ORACLE_DEV = "cuda"


def report(name, **values):
    print("PARITY " + json.dumps({"test": name, **values}))


def errors(got, ref):
    return {"max_rel": G.relmax(got, ref), "rel_fro": G.relfro(got, ref)}


@functools.lru_cache(maxsize=None)
def geometry(name):
    """(D, encoder, fp32 init params, oracle tables)."""
    D, R, V, NR, L = GEOMETRIES[name]
    _, enc = GE.make_geometry(R, V, NR, L, seed=0)
    return D, enc, O.init_params(V, NR, L, D, seed=1), G.tables(enc)


_MODELS = {}


def model(name, precision, compact, cta_group):
    """One model per (geometry, precision), its handle switched to the layout / cta_group of the case."""
    key = (name, precision)
    if key not in _MODELS:
        D, enc, params, _ = geometry(name)
        m = S.FCGGNN(enc, D, backbone=None, precision=precision)
        res = m.load_state_dict(params, strict=False)
        assert not res.unexpected_keys and not res.missing_keys
        _MODELS[key] = m.cuda()
    m = _MODELS[key]
    eng = m._engine_for(torch.device("cuda", torch.cuda.current_device()))
    eng.set_compact_rows(compact)
    eng.set_cta_group(cta_group)
    m.zero_grad(set_to_none=True)
    m.dropout_masks = None
    return m.eval()


def batch(name, size, seed):
    """size "1": one image of a verb with R roles; "cross": geometry.crossing_verbs (asserted to cross)."""
    D, enc, _, _ = geometry(name)
    R = enc.get_max_role_count()
    if size == "1":
        verbs = torch.tensor(GE.verbs_with_count(enc, R)[:1])
    else:
        verbs = GE.crossing_verbs(enc)
        counts = GE.verb_counts(enc)[verbs.numpy()]
        if R > 1:
            assert GE.straddles(counts), counts
        else:
            assert GE.compact_rows(counts)[1] > 256
        assert D < 1024 or len(verbs) <= 64
    return GE.make_batch(enc, len(verbs), D, seed, gt_verb=verbs)


def keep_masks(B, R, D, seed):
    g = torch.Generator().manual_seed(seed)
    return tuple(torch.rand(n, D, generator=g) < 0.5 for n in (B, B * R, B * R))


CASES = [(g, lay, cg, size) for g in GEOMETRIES for lay in LAYOUTS for cg in (2, 1) for size in ("1", "cross")]


def case_id(c):
    return "%s-%s-cg%d-B%s" % c


# ---------------------------------------------------------------------------------------------- fp32 forward
@pytest.mark.parametrize("name,layout,cta_group,size", CASES, ids=[case_id(c) for c in CASES])
def test_fp32_forward_vs_oracle(name, layout, cta_group, size):
    """precision="fp32", eval: verb logits and both noun-logit paths <= 1e-4 of max|ref| against fp64 (the predicted-
    verb path conditioned on the CUDA verbs), the same argmax on >= 99.9 % of the rows; the rows that differ must be
    near ties (fp64 top-1 / top-2 margin within twice the error bound)."""
    D, enc, params, (t, c) = geometry(name)
    m = model(name, "fp32", LAYOUTS[layout], cta_group)
    fv, fn, gt_verb, _ = batch(name, size, seed=11)
    with torch.no_grad():
        outs = m(fv.cuda(), gt_verb.cuda(), img_nouns=fn.cuda())
        p64 = {k: v.to(ORACLE_DEV, torch.float64) for k, v in params.items()}
        refs = O.forward(p64, fv.to(ORACLE_DEV, torch.float64), fn.to(ORACLE_DEV, torch.float64),
                         gt_verb.to(ORACLE_DEV), t, c, pred_verbs=outs[0].argmax(-1).to(ORACLE_DEV))
    res = {}
    for key, got, ref in zip(("verb", "pred_nouns", "gt_nouns"), outs, refs):
        got, ref = got.double().cpu().reshape(-1, ref.shape[-1]), ref.cpu().reshape(-1, ref.shape[-1])
        top2 = ref.topk(2, -1).values
        tie = (top2[:, 0] - top2[:, 1]) <= 2 * FP32_TOL * float(ref.abs().max())
        flips = got.argmax(-1) != ref.argmax(-1)
        res[key] = {**errors(got, ref), "rows": int(ref.shape[0]), "argmax_flips": int(flips.sum()),
                    "near_ties": int(tie.sum())}
        assert not (flips & ~tie).any(), (key, res[key])
    report("geometry_fp32_forward[%s]" % case_id((name, layout, cta_group, size)), errors=res)
    for key, e in res.items():
        assert e["max_rel"] <= FP32_TOL, (key, e)
        assert e["argmax_flips"] <= 1e-3 * e["rows"], (key, e)


# ---------------------------------------------------------------------------------------------- bf16 training step
def train_step(name, layout, cta_group, size, seed=7):
    """The CUDA training step (train mode, explicit keep masks, features as leaves): logits, losses, {param: grad},
    (dfeat_v, dfeat_n) and the inputs."""
    D, enc, params, _ = geometry(name)
    R = enc.get_max_role_count()
    m = model(name, "bf16", LAYOUTS[layout], cta_group).train()
    fv, fn, gt_verb, gt_nouns = batch(name, size, seed=seed)
    keeps = keep_masks(fv.shape[0], R, D, seed)
    m.dropout_masks = tuple(k.to(torch.uint8).cuda() for k in keeps)
    xv, xn = fv.cuda().requires_grad_(True), fn.cuda().requires_grad_(True)
    gv, gn = gt_verb.cuda(), gt_nouns.cuda()
    mpv, mpn, mgpn = m(xv, gv, img_nouns=xn)
    lv, ln, lg = m.verb_loss(mpv, gv), m.nouns_loss(mpn, gn), m.nouns_loss(mgpn, gn)
    (lv + ln).backward()
    grads = {k: (p.grad if p.grad is not None else torch.zeros_like(p)).detach().clone()
             for k, p in m.named_parameters()}
    m.dropout_masks = None
    logits = tuple(x.detach().clone() for x in (mpv, mpn, mgpn))
    return logits, (lv.item(), ln.item(), lg.item()), grads, (xv.grad, xn.grad), (fv, fn, gt_verb, gt_nouns), keeps


@pytest.mark.parametrize("name,layout,cta_group,size", CASES, ids=[case_id(c) for c in CASES])
def test_training_step_vs_oracle(name, layout, cta_group, size):
    """verb_loss + nouns_loss backward in train mode with explicit keep masks, the oracle's predicted-verb path
    conditioned on the CUDA verbs: the three logits, the three losses, all 20 gradients and dL/dfeat of both features.
    The padding row of role_emb gets exactly zero gradient."""
    D, enc, params, tabs = geometry(name)
    (mpv, mpn, mgpn), losses, grads, (dfv_c, dfn_c), b, keeps = train_step(name, layout, cta_group, size)
    (vl, nl, gl), ref, (pv, pn, gpn), (dfv, dfn) = G.oracle_step(
        params, b, tabs, mpv.argmax(-1).cpu(), keeps, True, device=ORACLE_DEV, num_labels=enc.get_num_labels())
    logits = {"verb": errors(mpv, pv), "pred_nouns": errors(mpn, pn), "gt_nouns": errors(mgpn, gpn)}
    gerr = {k: errors(grads[k], ref[k]) for k in ref}
    ferr = {"feat_v": errors(dfv_c, dfv), "feat_n": errors(dfn_c, dfn)}
    lref = [float(vl), float(nl), float(gl)]
    report("geometry_training_step[%s]" % case_id((name, layout, cta_group, size)), B=int(b[0].shape[0]),
           logits=logits, losses={"cuda": list(losses), "oracle": lref}, grads=gerr, feat_grads=ferr)
    for k, e in logits.items():
        assert e["max_rel"] <= LOGIT_TOL, (k, e)
    for mine, want in zip(losses, lref):
        assert abs(mine - want) <= LOSS_TOL * abs(want), (losses, lref)
    for k, e in {**gerr, **ferr}.items():
        assert e["max_rel"] <= GRAD_TOL, (k, e)
    assert float(grads["role_emb.weight"][enc.get_num_roles()].abs().max()) == 0.0


@pytest.mark.parametrize("cta_group", [2, 1])
@pytest.mark.parametrize("name", list(GEOMETRIES))
def test_compact_rows_equal_one_row_per_slot(name, cta_group):
    """The same training step on both row layouts, on the crossing batch: bit-identical logits, gradients (and
    dL/dfeat) within 2e-3 of max| | (the order of the sums differs)."""
    a = train_step(name, "compact", cta_group, "cross", seed=9)
    b = train_step(name, "per_slot", cta_group, "cross", seed=9)
    same = [bool(torch.equal(x, y)) for x, y in zip(a[0], b[0])]
    gerr = {k: G.relmax(a[2][k], b[2][k]) for k in a[2]}
    gerr.update(feat_v=G.relmax(a[3][0], b[3][0]), feat_n=G.relmax(a[3][1], b[3][1]))
    report("geometry_compact_vs_per_slot[%s,cg%d]" % (name, cta_group), logits_equal=same, grads=gerr)
    assert all(same), same
    for k, e in gerr.items():
        assert e <= LAYOUT_TOL, (k, e)


# ---------------------------------------------------------------------------------------------- model.ggsnn
@pytest.mark.parametrize("cta_group", [2, 1])
@pytest.mark.parametrize("name", ["D512_R8", "D256_R1"])
def test_ggsnn_vs_oracle(name, cta_group):
    """GGSNN.forward on caller-supplied states and a random real-valued mask that requires grad, at R = kMaxR and at
    R = 1: the output, d hidden, d mask and the 14 GGSNN gradients for loss = (out * G).sum()."""
    D, enc, params, _ = geometry(name)
    R = enc.get_max_role_count()
    B = 40
    gen = torch.Generator().manual_seed(17)
    hidden = torch.randn(B * R, D, generator=gen).relu()
    mask = G.random_mask(B, R, seed=B)
    up = torch.randn(hidden.shape, generator=gen)
    m = model(name, "bf16", True, cta_group)
    h = hidden.cuda().requires_grad_(True)
    mk = mask.cuda().requires_grad_(True)
    out = m.ggsnn(h, mask=mk)
    (out * up.cuda()).sum().backward()
    o, dh, dm, dp = G.oracle_ggsnn(params, hidden, mask, up, device=ORACLE_DEV)
    got = {"out": out, "hidden_state": h.grad, "mask": mk.grad,
           **{k: p.grad for k, p in m.ggsnn.named_parameters()}}
    ref = {"out": o, "hidden_state": dh, "mask": dm, **dp}
    errs = {k: errors(got[k], ref[k]) for k in ref}
    report("geometry_ggsnn[%s,cg%d]" % (name, cta_group), errors=errs)
    assert errs["out"]["max_rel"] <= LOGIT_TOL, errs["out"]
    for k, e in errs.items():
        assert e["max_rel"] <= GRAD_TOL, (k, e)


# ---------------------------------------------------------------------------------------------- decodes
DECODE_CASES = [(g, lay, cg) for g in GEOMETRIES for lay in LAYOUTS for cg in (2, 1)]


def decode_batch(name, B):
    D, enc, _, _ = geometry(name)
    return GE.make_batch(enc, B, D, seed=21)


@functools.lru_cache(maxsize=None)
def topk_oracle(name, B, k, verbs_key):
    """tests/situations_oracle.py in fp64 on the CPU (shared by the layouts / cta_groups that decode the same verbs):
    fp64 verb logits, the oracle's top-k verbs and log-probs, and with the CUDA verbs its labels and label log-probs."""
    D, enc, params, (t, c) = geometry(name)
    fv, fn, _, _ = decode_batch(name, B)
    cv = torch.from_numpy(np.frombuffer(verbs_key, dtype=np.int64).reshape(B, k).copy())
    p64 = {key: v.double() for key, v in params.items()}
    with torch.no_grad():
        pv = O.predict_verb(p64, fv.double())
        ov, ovl, _, _, _ = oracle_situations(p64, fv.double(), fn.double(), k, t, c)
        _, _, ol, oll, _ = oracle_situations(p64, fv.double(), fn.double(), k, t, c, verbs=cv)
    return pv, ov, ovl, ol, oll


@pytest.mark.parametrize("name,layout,cta_group", DECODE_CASES, ids=["%s-%s-cg%d" % c for c in DECODE_CASES])
def test_decodes_vs_oracle(name, layout, cta_group):
    """fp32 mode.  Top-k decode (k = 5) against tests/situations_oracle.py in fp64: the verbs where the fp64 ranking has
    clear gaps, and with the oracle conditioned on the CUDA verbs the labels (where the slot's top-2 are apart), their
    log-probs and the scores.  n-best decode (n = min(16, n_labels), beam of 5 verbs) against tests/nbest_oracle.py on
    the path's own logits, as tests/test_nbest_gpu.py: the same list except at near ties, scores the fp32 slot-order
    sums bit for bit; and the n best label assignments of the verbs with R roles, where at R = 8 some listed situation
    takes a label of rank >= 1 in slot 7 (the low nibble of the rank packing)."""
    D, enc, params, (t, c) = geometry(name)
    R, L = enc.get_max_role_count(), enc.get_num_labels()
    m = model(name, "fp32", LAYOUTS[layout], cta_group)
    B, k = 48, 5
    fv, fn, _, _ = decode_batch(name, B)
    fvc, fnc = fv.cuda(), fn.cuda()
    counts = torch.from_numpy(GE.verb_counts(enc))
    # ---- top-k
    s = m.situations_from_features(fvc, fnc, k=k)
    cv = s.verbs.cpu()
    pv, ov, ovl, ol, oll = topk_oracle(name, B, k, cv.numpy().tobytes())
    srt = torch.sort(pv, dim=1, descending=True, stable=True).values[:, :k + 1]
    ok_v = ((srt[:, :-1] - srt[:, 1:]) >= 1e-4 * pv.abs().max().item()).all(1)
    ok_l = torch.ones(B, k, dtype=torch.bool)
    p64 = {key: v.to(ORACLE_DEV, torch.float64) for key, v in params.items()}
    with torch.no_grad():
        for j in range(k):
            nl = O.predict_nouns(p64, fn.to(ORACLE_DEV, torch.float64), cv[:, j], t, c).cpu()
            top2 = torch.topk(nl, 2, -1).values
            real = torch.arange(R)[None, :] < counts[cv[:, j]][:, None]
            ok_l[:, j] = ~(((top2[..., 0] - top2[..., 1]) < 1e-4 * nl.abs().max().item()) & real).any(1)
    verb_agree = (s.verbs.cpu() == ov).all(1)[ok_v].double().mean().item()
    label_agree = (s.labels.cpu() == ol).all(-1)[ok_l].double().mean().item()
    topk = {"clear_verb_rows": int(ok_v.sum()), "verb_agree": verb_agree, "clear_candidates": int(ok_l.sum()),
            "label_agree": label_agree,
            "verb_logp_err": (s.verb_logp.cpu().double() - ovl)[ok_v].abs().max().item() if ok_v.any() else 0.0,
            "label_logp_err": (s.label_logp.cpu().double() - oll)[ok_l].abs().max().item(),
            "score_err": (s.score.cpu().double() - (s.verb_logp.cpu().double() + oll.sum(-1)))[ok_l].abs().max().item()}
    # ---- n-best over a beam of predicted verbs
    n = min(16, L)
    nb, exact = m.nbest_situations_from_features(fvc, fnc, n=n, verb_beam=k)
    verbs, vlp, bound = beam(m, fvc, k)
    ids, lps = slot_lists(m, fnc, verbs, n)
    check_self_consistent(nb, ids, lps, verbs, counts)
    compared, total = compare(nb, oracle_lists(verbs, vlp.cpu(), ids, lps, counts, n), n, 1e-5, tie=1e-6)
    last = nb.score[:, n - 1]
    clear = (last - bound).abs() > 1e-5
    # ---- n-best label assignments of the verbs with R roles
    full = torch.tensor(GE.verbs_with_count(enc, R)[:2])
    given = full[torch.arange(B) % len(full)][:, None].cuda()
    ng, _ = m.nbest_situations_from_features(None, fnc, n=n, verbs=given)
    gids, glps = slot_lists(m, fnc, given, n)
    check_self_consistent(ng, gids, glps, given, counts)
    gcompared, gtotal = compare(ng, oracle_lists(given, None, gids, glps, counts, n), n, 1e-5, tie=1e-6)
    last_slot_raised = int((ng.labels[:, :, R - 1].cpu() != gids[:, 0, R - 1, :1]).sum())
    report("geometry_decodes[%s-%s-cg%d]" % (name, layout, cta_group), topk=topk,
           nbest={"n": n, "compared": compared, "positions": total, "given_compared": gcompared,
                  "given_positions": gtotal, "last_slot_rank_ge_1": last_slot_raised})
    assert ok_v.float().mean() >= 0.25 and verb_agree >= 0.999, topk
    assert ok_l.float().mean() >= 0.5 and label_agree >= 0.999, topk
    assert topk["verb_logp_err"] <= 1e-4 and topk["label_logp_err"] <= 1e-4 and topk["score_err"] <= 1e-3, topk
    assert compared >= 0.5 * total and gcompared >= 0.5 * gtotal, (compared, total, gcompared, gtotal)
    assert torch.equal(exact[clear], (last >= bound)[clear])
    assert last_slot_raised > 0
    m.check_verbs()


# ---------------------------------------------------------------------------------------------- R = 9
def test_nine_roles_refused():
    """An encoder with 9 roles per verb is refused on the model's first call, with a message naming R."""
    _, enc = GE.make_geometry(9, 12, 12, 20, seed=0)
    m = S.FCGGNN(enc, 256, backbone=None).cuda().eval()
    fv, fn, gt_verb, _ = GE.make_batch(enc, 4, 256, seed=1)
    with pytest.raises(_lib.SrgError, match="R=9"):
        with torch.no_grad():
            m(fv.cuda(), gt_verb.cuda(), img_nouns=fn.cuda())
