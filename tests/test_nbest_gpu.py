"""-m gpu: the n-best situation decode (srg_situation_nbest, FCGGNN.nbest_situations_from_features and the launcher's
--nbest_situations) on a B200, against the oracle of tests/nbest_oracle.py."""
import ctypes
import math
import os

import pytest
import torch

import situation_recognition_b200 as S
from oracle import ggnn_oracle as O
from tests import regimes
from tests.nbest_oracle import nbest_best_first, rank_lists
from situation_recognition_b200 import _lib
from situation_recognition_b200.synthetic import make_batch, make_train_json

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def enc():
    return S.imsitu_encoder(make_train_json(seed=0), verbose=False)


@pytest.fixture(scope="module")
def tables(enc):
    return O.build_tables(enc.roles_per_verb, enc.verb_list, enc.role_list)


@pytest.fixture(scope="module")
def counts(enc):
    return torch.tensor([enc.get_role_count(v) for v in range(enc.get_num_verbs())])


def make_model(enc, D, precision, seed=0, compact=True, cta_group=2, params=None):
    if params is None:
        params = O.init_params(enc.get_num_verbs(), enc.get_num_roles(), enc.get_num_labels(), D, seed=seed)
    m = S.FCGGNN(enc, D, backbone=None, precision=precision)
    m.load_state_dict(params, strict=False)
    m = m.cuda().eval()
    eng = m._engine_for(torch.device("cuda", torch.cuda.current_device()))
    eng.set_compact_rows(compact)
    eng.set_cta_group(cta_group)
    return m, params


def topk_call(x, ldl, rows, n, k):
    lib = _lib.load()
    idx = torch.empty(rows, k, dtype=torch.int64, device="cuda")
    logp = torch.empty(rows, k, dtype=torch.float32, device="cuda")
    _lib.check(lib.srg_topk_logsoftmax(_lib.ptr(x), ldl, rows, n, k, _lib.ptr(idx), _lib.ptr(logp), _lib.stream_ptr()))
    return idx, logp


def padded(x, ldl):
    """x [rows, n] -> [rows, ldl] with x in the first n columns: the row layout the decode reads."""
    out = torch.zeros(x.shape[0], ldl, dtype=torch.float32, device="cuda")
    out[:, :x.shape[1]] = x
    return out


def beam(m, fv, kv):
    """The decode's candidate verbs [B, kv], their log-probs and the (kv+1)-th verb's log-prob, from predict_verb's
    logits through the same row kernel on the same row layout."""
    eng = m._engine_for(fv.device)
    B = fv.shape[0]
    with torch.no_grad():
        pv = padded(m.predict_verb(fv, B), eng.Vpad)
    idx, logp = topk_call(pv, eng.Vpad, B, eng.V, kv + 1)
    return idx[:, :kv].contiguous(), logp[:, :kv].contiguous(), logp[:, kv].contiguous()


def slot_lists(m, fn, verbs, n):
    """Per-slot top-n (label ids, log-probs) [B, kv, R, n] of these candidates, from predict_nouns' logits through the
    row kernel on the decode's row layout."""
    eng = m._engine_for(fn.device)
    B, kv = verbs.shape
    with torch.no_grad():
        nl = m.predict_nouns(fn.repeat_interleave(kv, 0), verbs.reshape(-1), B * kv)            # [B*kv, R, L]
    idx, logp = topk_call(padded(nl.reshape(-1, eng.L), eng.Lpad), eng.Lpad, B * kv * eng.R, eng.L, n)
    return idx.reshape(B, kv, eng.R, n).cpu(), logp.reshape(B, kv, eng.R, n).cpu()


def oracle_lists(verbs, vlp, ids, lps, counts, n):
    """Per image the oracle's n + 1 best as (score, verb, labels tuple); ids / lps [B, kv, R, m] in rank order."""
    verbs = verbs.cpu()
    B, kv = verbs.shape
    R = ids.shape[2]
    out = []
    for b in range(B):
        cands = []
        for j in range(kv):
            nr = int(counts[verbs[b, j]])
            cands.append((None if vlp is None else vlp[b, j].numpy()[()], lps[b, j, :nr].numpy()))
        rows = []
        for s, j, ranks in nbest_best_first(cands, n + 1):
            lab = [int(ids[b, j, r, k]) for r, k in enumerate(ranks)] + [-1] * (R - len(ranks))
            rows.append((float(s), int(verbs[b, j]), tuple(lab)))
        out.append(rows)
    return out


def compare(s, ref, n, rel, tie=None, rows=None):
    """The decode's list against the oracle's, image by image: the scores agree within `rel` (relative, at least 1
    absolute unit of rel) at every position, and at every position whose oracle score is more than `tie` (relative,
    default rel) from its neighbours' (no near-tie, the (n+1)-th included) the verb and labels are the oracle's.
    Returns (compared, positions)."""
    verbs, labels, score = s.verbs.cpu(), s.labels.cpu(), s.score.cpu().double()
    rows = range(len(ref)) if rows is None else rows
    tie = rel if tie is None else tie
    compared = total = 0
    for b, rb in zip(rows, ref):
        sc = [e[0] for e in rb]
        for i in range(n):
            tol = rel * max(1.0, abs(sc[i]))
            assert abs(score[b, i].item() - sc[i]) <= tol, (b, i, score[b, i].item(), sc[i])
            total += 1
            near = tie * max(1.0, abs(sc[i]))
            if (i > 0 and sc[i - 1] - sc[i] <= near) or (i + 1 < len(sc) and sc[i] - sc[i + 1] <= near):
                continue
            compared += 1
            assert (int(verbs[b, i]), tuple(labels[b, i].tolist())) == rb[i][1:], (b, i)
    return compared, total


def check_self_consistent(s, ids, lps, verbs_in, counts):
    """Each entry's labels come from its candidate's slot lists with their log-probs, pad slots are -1 / 0, and the
    score is verb_logp + label_logp summed in fp32 in slot order, bit for bit."""
    B, n, R = s.labels.shape
    acc = torch.zeros(B, n) if s.verb_logp is None else s.verb_logp.cpu().clone()
    lp = s.label_logp.cpu()
    for r in range(R):
        acc = acc + lp[:, :, r]                   # fp32, one add per slot (pad slots add 0)
    assert torch.equal(acc, s.score.cpu())
    real = torch.arange(R)[None, None, :] < counts[s.verbs.cpu()][:, :, None]
    assert (s.labels.cpu()[~real] == -1).all() and (lp[~real] == 0).all()
    assert (lp[real] <= 0).all()
    assert (s.verbs.cpu()[:, :, None] == verbs_in.cpu()[:, None, :]).any(-1).all()


def test_label_logp_never_positive():
    """The certificate needs every label log-prob <= 0: the row kernel's (x - M) - log S, with the max column's
    exp(0) in S.  One dominant column (S rounds to 1, its log-prob is exactly 0) and all-equal columns."""
    n, rows = 2001, 64
    x = torch.randn(rows, 2048, device="cuda")
    x[:32, 7] = 1e4
    x[32:, :n] = 3.25
    idx, logp = topk_call(x, 2048, rows, n, 16)
    assert (logp <= 0).all()
    assert (logp[:32, 0] == 0).all() and (idx[:32, 0] == 7).all()
    assert torch.equal(idx[32:], torch.arange(16, device="cuda").expand(32, 16))
    assert (logp[32:] - (-math.log(n))).abs().max().item() <= 1e-6


# ---------------------------------------------------------------------------------------------- 1. vs the oracle
_MODELS = {}


def cached_model(enc, precision, compact, cta_group):
    key = (precision, compact, cta_group)
    if key not in _MODELS:
        _MODELS[key] = make_model(enc, 256, precision, seed=1, compact=compact, cta_group=cta_group)[0]
    return _MODELS[key]


@pytest.mark.parametrize("cta_group", [2, 1])
@pytest.mark.parametrize("compact", [True, False])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("kv,n", [(kv, n) for kv in (1, 5, 15) for n in (1, 5, 16)])
def test_vs_oracle_on_own_logits(enc, counts, kv, n, precision, compact, cta_group):
    m = cached_model(enc, precision, compact, cta_group)
    B = 64
    fv, fn, _, _ = make_batch(enc, B, 256, seed=20 + kv + n, device="cuda")
    s, exact = m.nbest_situations_from_features(fv, fn, n=n, verb_beam=kv)
    assert s.verbs.shape == (B, n) and s.labels.shape == (B, n, enc.get_max_role_count()) and exact.dtype == torch.bool
    verbs, vlp, bound = beam(m, fv, kv)
    ids, lps = slot_lists(m, fn, verbs, n)
    check_self_consistent(s, ids, lps, verbs, counts)
    ref = oracle_lists(verbs, vlp.cpu(), ids, lps, counts, n)
    compared, total = compare(s, ref, n, 1e-5, tie=1e-6)
    print("n-best vs oracle (kv = %d, n = %d): %d of %d positions compared, the rest near ties" % (kv, n, compared,
                                                                                                  total))
    assert compared >= 0.5 * total, (compared, total)
    last = s.score[:, n - 1]
    clear = (last - bound).abs() > 1e-5
    assert torch.equal(exact[clear], (last >= bound)[clear])
    m.check_verbs()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("kv", [1, 5, 15])
def test_one_best_is_the_best_topk_candidate(enc, kv, precision):
    """n = 1 is the best-scoring candidate of situations_from_features(k=kv) (ties to the lower candidate), bit for
    bit: verb, verb log-prob, labels, label log-probs and score."""
    m = cached_model(enc, precision, True, 2)
    fv, fn, _, _ = make_batch(enc, 256, 256, seed=31, device="cuda")
    s, _ = m.nbest_situations_from_features(fv, fn, n=1, verb_beam=kv)
    t = m.situations_from_features(fv, fn, k=kv)
    j = torch.sort(t.score, dim=1, descending=True, stable=True).indices[:, :1]
    assert torch.equal(s.verbs, t.verbs.gather(1, j))
    assert torch.equal(s.verb_logp, t.verb_logp.gather(1, j))
    assert torch.equal(s.score, t.score.gather(1, j))
    R = t.labels.shape[2]
    assert torch.equal(s.labels, t.labels.gather(1, j[:, :, None].expand(-1, -1, R)))
    assert torch.equal(s.label_logp, t.label_logp.gather(1, j[:, :, None].expand(-1, -1, R)))


def test_fp32_vs_fp64_oracle(enc, tables, counts):
    B, D, kv, n = 64, 256, 5, 5
    params = O.init_params(enc.get_num_verbs(), enc.get_num_roles(), enc.get_num_labels(), D, seed=2,
                           dtype=torch.float64)
    m, _ = make_model(enc, D, "fp32", params=params)
    fv, fn, _, _ = make_batch(enc, B, D, seed=32)
    s, _ = m.nbest_situations_from_features(fv.cuda(), fn.cuda(), n=n, verb_beam=kv)
    verbs, _, _ = beam(m, fv.cuda(), kv)           # the oracle is conditioned on the decode's candidate verbs
    t, c = tables
    fv64, fn64 = fv.double(), fn.double()
    vlp = torch.log_softmax(O.predict_verb(params, fv64), 1).gather(1, verbs.cpu())
    ids = torch.empty(B, kv, enc.get_max_role_count(), n, dtype=torch.int64)
    lps = torch.empty(ids.shape, dtype=torch.float64)
    for j in range(kv):
        nl = O.predict_nouns(params, fn64, verbs[:, j].cpu(), t, c)
        ids[:, j], lps[:, j] = rank_lists(torch.log_softmax(nl, -1), n)
    ref = oracle_lists(verbs, vlp, ids, lps, counts, n)
    compared, total = compare(s, ref, n, 2e-4)
    print("n-best fp32 vs fp64: %d of %d positions compared, the rest near ties" % (compared, total))
    assert compared >= 0.2 * total        # at init the label distributions are flat: many situations lie within 2e-4


# ---------------------------------------------------------------------------------------------- 2. certificate
@pytest.mark.parametrize("regime", ["init", "peaked"])
def test_certificate_against_all_verbs(enc, tables, counts, regime):
    B, D, kv, n = 32, 256, 5, 5
    params = O.init_params(enc.get_num_verbs(), enc.get_num_roles(), enc.get_num_labels(), D, seed=3)
    batch = make_batch(enc, B, D, seed=33)
    params, (fv, fn, _, _) = regimes.REGIMES[regime](params, batch, tables)
    m, _ = make_model(enc, D, "bf16", params=params)
    fv, fn = fv.cuda(), fn.cuda()
    s, exact = m.nbest_situations_from_features(fv, fn, n=n, verb_beam=kv)
    V = enc.get_num_verbs()
    # every verb, in the decode's order, with the row kernel's log-probs for the beam and fp32 log-softmax beyond it
    verbs, vlp, _ = beam(m, fv, kv)
    with torch.no_grad():
        pv = m.predict_verb(fv, B)
    order = torch.sort(pv, dim=1, descending=True, stable=True).indices
    assert torch.equal(order[:, :kv], verbs)
    all_lp = torch.log_softmax(pv, 1).gather(1, order)
    all_lp[:, :kv] = vlp
    ids, lps = [], []
    for c0 in range(0, V, 16):                     # the role graphs of all verbs, 16 candidates at a time
        i, l = slot_lists(m, fn, order[:, c0:c0 + 16].contiguous(), n)
        ids.append(i)
        lps.append(l)
    ref = oracle_lists(order, all_lp.cpu(), torch.cat(ids, 1), torch.cat(lps, 1), counts, n)
    rows = [b for b in range(B) if exact[b]]
    compared, total = compare(s, [ref[b] for b in rows], n, 1e-5, tie=1e-6, rows=rows)
    frac = exact.float().mean().item()
    print("n-best certificate (%s, kv = %d, n = %d): %.3f of the images certified; %d of %d of their positions "
          "compared, the rest near ties" % (regime, kv, n, frac, compared, total))
    if regime == "peaked":
        assert frac >= 0.5
    assert compared >= 0.5 * total


# ---------------------------------------------------------------------------------------------- 3. given verbs
def test_given_verbs(enc, counts):
    m = cached_model(enc, "bf16", True, 2)
    B, n = 64, 6
    fv, fn, gt_verb, _ = make_batch(enc, B, 256, seed=34, device="cuda")
    pair = torch.stack([gt_verb, (gt_verb + 7) % enc.get_num_verbs()], 1)
    s2c, exact = m.nbest_situations_from_features(None, fn, n=n, verbs=pair)
    assert s2c.verb_logp is None and exact.all()
    ids, lps = slot_lists(m, fn, pair, n)
    check_self_consistent(s2c, ids, lps, pair, counts)
    compared, total = compare(s2c, oracle_lists(pair, None, ids, lps, counts, n), n, 1e-5, tie=1e-6)
    assert compared >= 0.5 * total, (compared, total)
    # a repeated candidate: candidate 2 has candidate 0's inputs, so each of its situations ties exactly with a twin of
    # candidate 0 and ranks right after it (lower candidate first).  The list is the two-candidate list with those
    # twins merged in by (score, candidate), bit for bit.
    verbs = torch.cat([pair, gt_verb[:, None]], 1)
    s, exact = m.nbest_situations_from_features(None, fn, n=n, verbs=verbs)
    assert s.verb_logp is None and exact.all()
    for b in range(B):
        rows = [(float(s2c.score[b, i]), 0 if int(s2c.verbs[b, i]) == int(gt_verb[b]) else 1, i) for i in range(n)]
        rows += [(sc, 2, i) for sc, j, i in rows if j == 0]
        order = [i for _, _, i in sorted(rows, key=lambda e: (-e[0], e[1]))[:n]]
        for got, ref in ((s.verbs, s2c.verbs), (s.labels, s2c.labels), (s.label_logp, s2c.label_logp),
                         (s.score, s2c.score)):
            assert torch.equal(got[b], ref[b, order]), b
    s1, _ = m.nbest_situations_from_features(None, fn, n=n, verbs=gt_verb[:, None])
    assert (s1.verbs == gt_verb[:, None]).all()
    m.train()                                          # no dropout and no autograd node in train mode either
    s2, _ = m.nbest_situations_from_features(None, fn, n=n, verbs=verbs)
    m.eval()
    assert not s2.score.requires_grad
    for a, b in zip(s2, s):
        assert a is None and b is None or torch.equal(a, b)
    for kw in (dict(n=0), dict(n=17), dict(verb_beam=0), dict(verb_beam=16)):
        with pytest.raises(_lib.SrgError):
            m.nbest_situations_from_features(fv, fn, **kw)


# ---------------------------------------------------------------------------------------------- 4. reproducibility
def test_repeatable_and_cuda_graph_replay(enc):
    m = cached_model(enc, "bf16", True, 2)
    B = 512
    fv, fn, _, _ = make_batch(enc, B, 256, seed=35, device="cuda")
    a, ea = m.nbest_situations_from_features(fv, fn, n=16, verb_beam=15)
    b, eb = m.nbest_situations_from_features(fv, fn, n=16, verb_beam=15)
    for x, y in zip(a + (ea,), b + (eb,)):
        assert torch.equal(x, y)
    sv, sn = fv.clone(), fn.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        m.nbest_situations_from_features(sv, sn, n=5)          # packs the weights before the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out, ex = m.nbest_situations_from_features(sv, sn, n=5)
    for seed in (36, 37):
        nv, nn_, _, _ = make_batch(enc, B, 256, seed=seed, device="cuda")
        sv.copy_(nv)
        sn.copy_(nn_)
        g.replay()
        eager, ee = m.nbest_situations_from_features(nv, nn_, n=5)
        for x, y in zip(out + (ex,), eager + (ee,)):
            assert torch.equal(x, y)


def nbest_call(eng, m, fn, verbs, vlp, bound, n, ws, ws_bytes, prec=0, outs=None, kv=None):
    B = verbs.shape[0]
    kv = verbs.shape[1] if kv is None else kv
    o = outs or dict(verbs=torch.empty(B, n, dtype=torch.int64, device="cuda"),
                     vlp=torch.empty(B, n, device="cuda"),
                     labels=torch.empty(B, n, eng.R, dtype=torch.int64, device="cuda"),
                     lp=torch.empty(B, n, eng.R, device="cuda"), score=torch.empty(B, n, device="cuda"),
                     exact=torch.empty(B, dtype=torch.bool, device="cuda"))
    rc = eng.lib.srg_situation_nbest(eng.h, _lib.ptr(fn), _lib.ptr(verbs), B, kv, _lib.ptr(m.role_emb.weight),
                                     _lib.ptr(m.verb_emb.weight), _lib.ptr(vlp), _lib.ptr(bound), n,
                                     _lib.ptr(o["verbs"]), _lib.ptr(o["vlp"]), _lib.ptr(o["labels"]), _lib.ptr(o["lp"]),
                                     _lib.ptr(o["score"]), _lib.ptr(o["exact"]), prec, ws, ws_bytes, eng.stream())
    return rc, o


def test_workspace_at_any_16_byte_offset(enc):
    m = cached_model(enc, "bf16", True, 2)
    B, kv, n = 96, 5, 16
    fv, fn, _, _ = make_batch(enc, B, 256, seed=38, device="cuda")
    ref, ref_exact = m.nbest_situations_from_features(fv, fn, n=n, verb_beam=kv)
    eng = m._engine_for(fn.device)
    verbs, vlp, bound = beam(m, fv, kv)
    need = eng.lib.srg_situation_nbest_workspace_bytes(eng.h, B, kv, n, 0)
    assert need > eng.lib.srg_situation_workspace_bytes(eng.h, B, kv, 0)
    buf = torch.empty(need + 2048, dtype=torch.uint8, device="cuda")
    base = (-buf.data_ptr()) % 1024
    for extra in (0, 512, 16, 1008):
        buf.fill_(0xFF)
        rc, o = nbest_call(eng, m, fn, verbs, vlp, bound, n, ctypes.c_void_p(buf.data_ptr() + base + extra), need)
        _lib.check(rc)
        got = (o["verbs"], o["vlp"], o["labels"], o["lp"], o["score"])
        for x, y in zip(got, ref):
            assert torch.equal(x, y), extra
        assert torch.equal(o["exact"], ref_exact)


def test_large_batch_finite_and_sampled_vs_oracle(enc, counts):
    m, _ = make_model(enc, 2048, "bf16", seed=4)
    B, kv, n = 6144, 5, 5
    fv, fn, _, _ = make_batch(enc, B, 2048, seed=39, device="cuda")
    s, exact = m.nbest_situations_from_features(fv, fn, n=n, verb_beam=kv)
    assert torch.isfinite(s.score).all() and torch.isfinite(s.verb_logp).all() and torch.isfinite(s.label_logp).all()
    rows = torch.randperm(B, generator=torch.Generator().manual_seed(5))[:64].tolist()
    verbs, vlp, bound = beam(m, fv[rows], kv)
    ids, lps = slot_lists(m, fn[rows], verbs, n)
    ref = oracle_lists(verbs, vlp.cpu(), ids, lps, counts, n)
    compared, total = compare(s, ref, n, 1e-5, tie=1e-6, rows=rows)
    assert compared >= 0.5 * total, (compared, total)
    last = s.score[rows, n - 1]
    clear = (last - bound).abs() > 1e-5
    assert torch.equal(exact[rows][clear], (last >= bound)[clear])
    m.check_verbs()


# ---------------------------------------------------------------------------------------------- 5. refusals
def test_refusals_on_a_live_handle(enc):
    m = cached_model(enc, "bf16", True, 2)
    B, kv, n = 8, 3, 4
    fv, fn, _, _ = make_batch(enc, B, 256, seed=40, device="cuda")
    m.nbest_situations_from_features(fv, fn, n=n, verb_beam=kv)
    eng = m._engine_for(fn.device)
    verbs, vlp, bound = beam(m, fv, kv)
    need = eng.lib.srg_situation_nbest_workspace_bytes(eng.h, B, 16, 16, 0)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    wsp = ctypes.c_void_p(ws.data_ptr())
    torch.cuda.synchronize()
    before = eng.lib.srg_launch_count()
    for bad_kv, bad_n in ((0, n), (17, n), (kv, 0), (kv, 17)):
        v = torch.zeros(B, max(bad_kv, 1), dtype=torch.int64, device="cuda")
        rc, _ = nbest_call(eng, m, fn, v, None, None, bad_n, wsp, need, kv=bad_kv)
        assert rc != 0
    _, outs = nbest_call(eng, m, fn, verbs, vlp, bound, n, wsp, need)
    after_ok = eng.lib.srg_launch_count()
    assert after_ok > before
    for key in ("verbs", "labels", "lp", "score"):
        o = dict(outs)
        o[key] = None
        rc, _ = nbest_call(eng, m, fn, verbs, vlp, bound, n, wsp, need, outs=o)
        assert rc != 0 and b"null argument" in eng.lib.srg_last_error()
    short = eng.lib.srg_situation_nbest_workspace_bytes(eng.h, B, kv, n, 0) - 1
    rc, _ = nbest_call(eng, m, fn, verbs, vlp, bound, n, wsp, short)
    assert rc != 0 and b"workspace too small" in eng.lib.srg_last_error()
    rc, _ = nbest_call(eng, m, fn, verbs, vlp, bound, n, None, need)
    assert rc != 0
    rc, _ = nbest_call(eng, m, fn, verbs, vlp, bound, n, wsp, need, prec=1)          # weights packed for bf16
    assert rc != 0
    # a handle whose role tables were never set
    h = ctypes.c_void_p()
    _lib.check(eng.lib.srg_create(ctypes.byref(h), torch.cuda.current_device(), 256, eng.R, 4, eng.V, eng.NR, eng.L))
    try:
        bare = type("E", (), dict(lib=eng.lib, h=h, R=eng.R, stream=eng.stream))()
        rc, _ = nbest_call(bare, m, fn, verbs, vlp, bound, n, wsp, need)
        assert rc != 0 and b"srg_set_tables" in eng.lib.srg_last_error()
    finally:
        eng.lib.srg_destroy(h)
    assert eng.lib.srg_launch_count() == after_ok


# ---------------------------------------------------------------------------------------------- 6. launcher
def _lines(out, start):
    lines = [l for l in out.splitlines() if l.strip()]
    return lines[[i for i, l in enumerate(lines) if l.startswith(start)][0]:]


def test_launcher_nbest_situations(tmp_path, capsys, monkeypatch):
    from situation_recognition_b200 import sr
    from tests.test_launcher import _make_dataset
    first = _make_dataset(str(tmp_path))
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("SRG_SEED", "7")
    common = ["--no_pretrained", "--num_workers", "0", "--batch_size", "4"]
    img = os.path.join("resized_256", first)
    sr.main(common + ["--test_img", img])
    base = _lines(capsys.readouterr().out, "Using ")
    sr.main(common + ["--test_img", img, "--nbest_situations", "4"])
    out = _lines(capsys.readouterr().out, "Using ")
    assert out[:len(base)] == base                       # the existing lines are unchanged
    heads = [l for l in out[len(base):] if l.startswith("situation ")]
    assert [h.split()[1] for h in heads] == ["1", "2", "3", "4"] and all("%)" in h for h in heads)
    scores = [float(h.rsplit("= ", 1)[1]) for h in heads]
    assert all(a >= b for a, b in zip(scores, scores[1:]))
    assert out[-1] in ("n-best list certified over all verbs: yes", "n-best list certified over all verbs: no")
    sr.main(common + ["--test_img", img, "--verb", "verb003", "--nbest_situations", "4"])
    out = capsys.readouterr().out.splitlines()
    heads = [l for l in out if l.startswith("situation ")]
    assert len(heads) == 4 and all("(given): verb003" in h for h in heads)
    assert out[-1] == "n-best list certified over all verbs: yes"
