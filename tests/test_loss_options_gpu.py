"""-m gpu: the loss options (class weights, label smoothing, "mean" / "sum" / "none") against
torch.nn.functional.cross_entropy in fp64.

  * the loss kernels on every output route: fp32 dlogits read three times (a clone), fp32 dlogits with the
    classifier's per-tile softmax statistics, and the bf16 operand the classifier's backward reads (side channel);
  * all-ones class weights (which select the option arithmetic) against the default-option kernels;
  * the training step with label smoothing and noun weights against an fp64 oracle step;
  * two ranks with unequal shards and class weights on both losses;
  * GraphedTrainStep with options: replay = eager, and replays are bit-identical.
"""
import ctypes
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import situation_recognition_b200 as S  # noqa: E402
from oracle import ggnn_oracle as O  # noqa: E402
from situation_recognition_b200 import _lib  # noqa: E402
from situation_recognition_b200.synthetic import make_batch, make_train_json  # noqa: E402
from tests import regimes as G  # noqa: E402

pytestmark = pytest.mark.gpu

V, L = 504, 2001
LOSS_TOL, DLOGITS_TOL = 1e-5, 1e-4           # the suite's loss-kernel bounds (test_saturation_gpu.py)
GRAD_TOL, LOGIT_TOL = 3e-2, 2e-2             # the suite's bf16 training-step bounds


def enc_syn():
    return S.imsitu_encoder(make_train_json(seed=0), verbose=False)


def model_from(params, enc, D):
    m = S.FCGGNN(enc, D, backbone=None, precision="bf16")
    res = m.load_state_dict(params, strict=False)
    assert not res.unexpected_keys and not res.missing_keys
    return m.cuda().eval()


def weights(kind, n, seed):
    """None, random positive, or positive with exact zeros (every third class, class 0 included)."""
    if kind is None:
        return None
    g = torch.Generator().manual_seed(seed)
    w = torch.rand(n, generator=g) * 2 + 0.1
    if kind == "zeros":
        w[::3] = 0
    return w.cuda()


def craft_targets(gt_verb, gt_nouns):
    """Image 0: every noun target ignored.  Annotation 2: every real target on class 0 (weight 0 under "zeros"), so its
    weighted denominator is 0."""
    gn = gt_nouns.clone()
    gn[0] = L
    a2 = gn[:, 2]
    a2[a2 != L] = 0
    return gt_verb.clone(), gn


def ref_loss(which, z, gt, w, eps, red):
    """torch's definition in fp64; nouns: summed over the 3 annotations, a zero "mean" denominator contributes 0."""
    w = None if w is None else w.double()
    if which == "verb":
        if red == "mean" and w is not None and float(w[gt].sum()) == 0:
            return (z * 0).sum()
        return F.cross_entropy(z, gt, weight=w, label_smoothing=eps, reduction=red)
    B, R, _ = z.shape
    zf = z.reshape(B * R, L)
    parts = []
    for a in range(3):
        y = gt[:, a].reshape(-1)
        if red == "none":
            parts.append(F.cross_entropy(zf, y, weight=w, ignore_index=L, label_smoothing=eps,
                                         reduction="none").view(B, R))
            continue
        valid = y != L
        den = float(valid.sum()) if w is None else float(w[y[valid]].sum())
        if red == "mean" and den == 0:
            continue
        parts.append(F.cross_entropy(zf, y, weight=w, ignore_index=L, label_smoothing=eps, reduction=red))
    return torch.stack(parts, 1) if red == "none" else sum(parts, (z * 0).sum())


def bf16_ulp(x):
    """One bf16 ulp at |x| (2^-133 for zero: the subnormal spacing)."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.pow(2.0, e - 7)


def _bf16_route(m, which, logits, gt, w, eps, red, upstream):
    """The side-channel operand: srg_*_loss_backward_ex with dlogits_bf16 and the classifier's softmax statistics."""
    eng = m._engine_for(logits.device)
    rows = logits.shape[0] * (logits.shape[1] if which == "nouns" else 1)
    npad = eng.Lpad if which == "nouns" else eng.Vpad
    dlb = torch.full((rows, npad), float("nan"), dtype=torch.bfloat16, device="cuda")
    red_code = _lib.SRG_REDUCTION[red]
    gpt = upstream.contiguous() if red == "none" else None
    gout = None if red == "none" else upstream.reshape(1).contiguous()
    o = _lib.SrgLossOpts(_lib.ptr(w), eps, red_code, None, _lib.ptr(gpt))
    st = ctypes.c_void_p(logits._srg_stats[1])
    B = logits.shape[0]
    if which == "nouns":
        counts = torch.empty(3, device="cuda")
        _lib.check(eng.lib.srg_count_targets_weighted(eng.h, _lib.ptr(gt), B, _lib.ptr(w), _lib.ptr(counts),
                                                      eng.stream()))
        _lib.check(eng.lib.srg_nouns_loss_backward_ex(eng.h, _lib.ptr(logits), npad, _lib.ptr(gt), B, _lib.ptr(counts),
                                                      _lib.ptr(gout), 1.0, None, _lib.ptr(dlb), 0, st,
                                                      ctypes.byref(o), eng.stream()))
    else:
        total = None
        if w is not None:
            total = torch.empty(1, device="cuda")
            _lib.check(eng.lib.srg_verb_weight_total(eng.h, _lib.ptr(gt), B, _lib.ptr(w), _lib.ptr(total),
                                                     eng.stream()))
        _lib.check(eng.lib.srg_verb_loss_backward_ex(eng.h, _lib.ptr(logits), npad, _lib.ptr(gt), B, 1.0 / B,
                                                     _lib.ptr(total), _lib.ptr(gout), 1.0, None, _lib.ptr(dlb), 0, st,
                                                     ctypes.byref(o), eng.stream()))
    return dlb


@pytest.mark.parametrize("regime", ["init", "peaked"])
@pytest.mark.parametrize("cg", [1, 2])
def test_loss_kernels_vs_torch_fp64(cg, regime):
    """Every (eps, weight, reduction) on the model's own logits, three routes, against F.cross_entropy in fp64: loss
    <= 1e-5 and fp32 dlogits <= 1e-4 relative to max; the bf16 operand within one bf16 ulp of the fp32 route's
    dlogits (with the softmax statistics), its padding columns 0.  "none" is back-propagated with a random per-target
    upstream gradient times per-image weights.  A zero denominator gives 0, never NaN."""
    D, B = 256, 24
    enc = enc_syn()
    params = O.init_params(V, 190, L, D, seed=0)
    batch = make_batch(enc, B, D, seed=5)
    params, batch = G.REGIMES[regime](params, batch, G.tables(enc))
    m = model_from(params, enc, D)
    m._engine_for(torch.device("cuda")).set_cta_group(cg)
    gv, gn = [x.cuda() for x in craft_targets(batch[2], batch[3])]
    with torch.no_grad():
        pv, pn, _ = m(batch[0].cuda(), gv, img_nouns=batch[1].cuda())
    gen = torch.Generator().manual_seed(7)
    worst = {}
    for which, logits, gt, n in (("verb", pv, gv, V), ("nouns", pn, gn, L)):
        assert logits._srg_stats is not None
        for eps in (0.0, 0.1, 1.0):
            for wk in (None, "rand", "zeros"):
                w = weights(wk, n, seed=11)
                for red in ("mean", "sum", "none"):
                    tag = (which, eps, wk, red)
                    shape = gt.shape if which == "nouns" else (B,)
                    per_image = torch.rand(B, generator=gen) + 0.5
                    up = (torch.rand(shape, generator=gen) * per_image.view(-1, *([1] * (len(shape) - 1)))).cuda() \
                        if red == "none" else torch.tensor(1.7, device="cuda")
                    z64 = logits.detach().double().requires_grad_(True)
                    ref = ref_loss(which, z64, gt, w, eps, red)
                    (ref * up.double()).sum().backward()
                    grads = {}
                    for route in ("three_pass", "stats"):
                        x = logits.detach().clone() if route == "three_pass" else logits.detach()
                        if route == "stats":
                            x._srg_stats = logits._srg_stats
                        x.requires_grad_(True)
                        call = m.verb_loss if which == "verb" else m.nouns_loss
                        got = call(x, gt, weight=w, label_smoothing=eps, reduction=red)
                        assert got.shape == ref.shape, tag
                        assert torch.isfinite(got).all(), tag
                        e_loss = G.relmax(got, ref) if ref.abs().max() > 0 else got.abs().max().item()
                        (got * up).sum().backward()
                        grads[route] = x.grad
                        e_dl = G.relmax(x.grad, z64.grad) if z64.grad.abs().max() > 0 else x.grad.abs().max().item()
                        worst[tag + (route,)] = (e_loss, e_dl)
                        assert e_loss <= LOSS_TOL, (tag, route, e_loss)
                        assert e_dl <= DLOGITS_TOL, (tag, route, e_dl)
                    dlb = _bf16_route(m, which, logits, gt, w, eps, red, up).float()
                    g32 = grads["stats"].reshape(dlb.shape[0], n)
                    assert torch.all(dlb[:, n:] == 0), tag
                    diff = (dlb[:, :n] - g32).abs()
                    assert torch.all(diff <= bf16_ulp(torch.maximum(g32.abs(), dlb[:, :n].abs()))), \
                        (tag, diff.max().item())
    e = max(worst.values(), key=lambda t: t[1])
    print("PARITY loss_options[cg=%d,%s]: %d cases, worst loss err %.2e, worst dlogits err %.2e" %
          (cg, regime, len(worst), max(v[0] for v in worst.values()), e[1]))


def test_zero_denominators_give_zero():
    """All targets at zero-weight classes: the weighted "mean" of both losses is 0 with a 0 gradient (torch: NaN)."""
    D, B = 256, 8
    enc = enc_syn()
    params = O.init_params(V, 190, L, D, seed=0)
    fv, fn, gv, gn = make_batch(enc, B, D, seed=5)
    m = model_from(params, enc, D)
    with torch.no_grad():
        pv, pn, _ = m(fv.cuda(), gv.cuda(), img_nouns=fn.cuda())
    wv, wn = torch.ones(V, device="cuda"), torch.ones(L, device="cuda")
    wv[gv] = 0
    gn = gn.cuda()
    wn[gn[gn != L]] = 0
    for x, call, gt, w in ((pv, m.verb_loss, gv.cuda(), wv), (pn, m.nouns_loss, gn, wn)):
        x = x.detach().clone().requires_grad_(True)
        loss = call(x, gt, weight=w, label_smoothing=0.1)
        loss.backward()
        assert loss.item() == 0.0 and torch.all(x.grad == 0)


def test_all_ones_weights_equal_the_defaults():
    """weight = ones selects the option arithmetic; its losses and fp32 gradients equal the default-option kernels'
    within fp32 rounding, and a training step's gradients (side channel) agree far inside the bf16 bounds."""
    D, B = 256, 24
    enc = enc_syn()
    params = O.init_params(V, 190, L, D, seed=0)
    fv, fn, gv, gn = [x.cuda() for x in make_batch(enc, B, D, seed=5)]
    ones_v, ones_n = torch.ones(V, device="cuda"), torch.ones(L, device="cuda")
    res = []
    for opt in (False, True):
        m = model_from(params, enc, D)
        kv = {"weight": ones_v} if opt else {}
        kn = {"weight": ones_n} if opt else {}
        pv, pn, gpn = m(fv, gv, img_nouns=fn)
        xs = [t.detach().clone().requires_grad_(True) for t in (pv, pn)]
        l32 = m.verb_loss(xs[0], gv, **kv) + m.nouns_loss(xs[1], gn, **kn)
        l32.backward()
        vl, nl, gl = m.verb_loss(pv, gv, **kv), m.nouns_loss(pn, gn, **kn), m.nouns_loss(gpn, gn, **kn)
        (vl + nl).backward()
        res.append((torch.stack([vl, nl, gl]).detach(), [x.grad for x in xs],
                    {k: p.grad.detach().clone() for k, p in m.named_parameters()}))
    (l0, d0, g0), (l1, d1, g1) = res
    assert torch.allclose(l0, l1, rtol=2e-6, atol=0), (l0, l1)
    for a, b in zip(d0, d1):
        assert G.relmax(b, a) <= 2e-6
    for k in g0:
        assert G.relmax(g1[k], g0[k]) <= 1e-3, k


def _oracle_step(params, batch, tabs, pred_verbs, verb_kw, nouns_kw):
    """fp64 autograd of the oracle's step with F.cross_entropy under the given options; dL/dfeat too."""
    dev = "cuda"
    ps = {k: v.double().to(dev).requires_grad_(True) for k, v in params.items()}
    fv, fn = (x.double().to(dev).requires_grad_(True) for x in batch[:2])
    gv, gn = batch[2].to(dev), batch[3].to(dev)
    t, c = tabs
    pv, pn, gpn = O.forward(ps, fv, fn, gv, t, c, pred_verbs=pred_verbs.to(dev))
    vl = ref_loss("verb", pv, gv, verb_kw.get("weight"), verb_kw.get("label_smoothing", 0.0), "mean")
    nl = ref_loss("nouns", pn, gn, nouns_kw.get("weight"), nouns_kw.get("label_smoothing", 0.0), "mean")
    gl = ref_loss("nouns", gpn, gn, nouns_kw.get("weight"), nouns_kw.get("label_smoothing", 0.0), "mean")
    (vl + nl).backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in ps.items()}
    return (vl, nl, gl), grads, (pv, pn, gpn), (fv.grad, fn.grad)


@pytest.mark.parametrize("compact", [True, False])
@pytest.mark.parametrize("D", [256, 2048])
def test_training_step_with_options_vs_fp64(D, compact):
    """sr.py's step with label smoothing 0.1 on both losses and class weights on the nouns: logits, losses, all 20
    gradients and dL/dfeat against the fp64 oracle step whose losses are F.cross_entropy with the same options."""
    B = 16
    enc = enc_syn()
    params = O.init_params(V, 190, L, D, seed=0)
    batch = make_batch(enc, B, D, seed=5)
    m = model_from(params, enc, D)
    m._engine_for(torch.device("cuda")).set_compact_rows(compact)
    wn = weights("rand", L, seed=3)
    vkw, nkw = {"label_smoothing": 0.1}, {"label_smoothing": 0.1, "weight": wn}
    fv, fn = (x.cuda().requires_grad_(True) for x in batch[:2])
    gv, gn = batch[2].cuda(), batch[3].cuda()
    pv, pn, gpn = m(fv, gv, img_nouns=fn)
    vl, nl, gl = m.verb_loss(pv, gv, **vkw), m.nouns_loss(pn, gn, **nkw), m.nouns_loss(gpn, gn, **nkw)
    (vl + nl).backward()
    (rvl, rnl, rgl), ref, (rpv, rpn, rgpn), (dfv, dfn) = _oracle_step(params, batch, G.tables(enc),
                                                                      pv.argmax(-1).cpu(), vkw, nkw)
    errs = {"logits": max(G.relmax(a, b) for a, b in ((pv, rpv), (pn, rpn), (gpn, rgpn)))}
    errs["losses"] = max(abs(a.item() - b.item()) / abs(b.item()) for a, b in ((vl, rvl), (nl, rnl), (gl, rgl)))
    for k, p in m.named_parameters():
        errs[k] = G.relmax(p.grad, ref[k])
    errs["dfeat_verbs"], errs["dfeat_nouns"] = G.relmax(fv.grad, dfv), G.relmax(fn.grad, dfn)
    print("PARITY loss_options_step[D=%d,compact=%s]: %s" % (D, compact, max(errs.items(), key=lambda kv: kv[1])))
    assert len([k for k, _ in m.named_parameters()]) == 20
    assert errs["logits"] <= LOGIT_TOL and errs["losses"] <= LOGIT_TOL, errs
    for k, e in errs.items():
        assert e <= GRAD_TOL, (k, e)


# ---------------------------------------------------------------------------------------------- two ranks
B2, D2 = 21, 256


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_setup():
    enc = enc_syn()
    params = O.init_params(V, 190, L, D2, seed=0)
    batch = make_batch(enc, B2, D2, seed=3)
    kw = ({"weight": weights("rand", V, 1), "label_smoothing": 0.1},
          {"weight": weights("zeros", L, 2), "label_smoothing": 0.1})
    return enc, params, batch, kw


def _rank_step(m, flat, batch, lo, hi, kw):
    fv, fn, gv, gn = [x[lo:hi].cuda() for x in batch]
    flat.zero()
    pv, pn, gpn = m(fv, gv, img_nouns=fn)
    vl, nl, gl = m.verb_loss(pv, gv, **kw[0]), m.nouns_loss(pn, gn, **kw[1]), m.nouns_loss(gpn, gn, **kw[1])
    (vl + nl).backward()
    return torch.stack([vl.detach(), nl.detach(), gl.detach()])


def _rank_worker(rank, world, port, out, know_global_batch):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from situation_recognition_b200 import parallel
    enc, params, batch, kw = _rank_setup()
    m = model_from(params, enc, D2)
    flat = parallel.attach(m)
    m.global_batch = B2 if know_global_batch else None
    lo, hi = parallel.shard_range(B2, rank, world)
    losses = _rank_step(m, flat, batch, lo, hi, kw)
    flat.all_reduce()
    dist.all_reduce(losses)
    torch.cuda.synchronize()
    if rank == 0:
        grads = {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters()}
        torch.save({"losses": losses.cpu(), "grads": grads},
                   out)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("know_global_batch", [False, True])
def test_two_ranks_with_class_weights_equal_full_batch(tmp_path, know_global_batch):
    """Unequal shards (11 + 10 images), class weights and smoothing on both losses: the weighted denominators are
    global (all-reduced on the stream; global_batch cannot stand in for a weighted one), so the summed shard losses and
    gradients equal the full batch's."""
    from situation_recognition_b200 import parallel
    out = str(tmp_path / "ranks.pt")
    mp.spawn(_rank_worker, args=(2, _free_port(), out, know_global_batch), nprocs=2, join=True)
    got = torch.load(out)
    enc, params, batch, kw = _rank_setup()
    m = model_from(params, enc, D2)
    flat = parallel.attach(m)
    losses = _rank_step(m, flat, batch, 0, B2, kw).cpu()
    assert torch.allclose(got["losses"], losses, rtol=2e-5, atol=1e-6), (got["losses"], losses)
    worst = 0.0
    for k, p in m.named_parameters():
        v = p.grad.detach().cpu()
        err = (got["grads"][k] - v).abs().max().item() / max(v.abs().max().item(), 1e-12)
        worst = max(worst, err)
        assert err <= 5e-3, (k, err)
    print("PARITY loss_options_two_ranks[global_batch=%s]: worst grad err %.2e" % (know_global_batch, worst))


# ---------------------------------------------------------------------------------------------- CUDA graph
def test_graphed_step_with_options():
    """GraphedTrainStep with smoothing and class weights: the replayed first step equals the eager one, and two replays
    from the same state give bit-identical losses (the weighted denominators and the option losses are summed in a
    fixed order)."""
    from situation_recognition_b200 import parallel
    from situation_recognition_b200.graph import GraphedTrainStep
    B, D = 24, 2048
    enc = enc_syn()
    params = O.init_params(V, 190, L, D, seed=0)
    batch = [x.cuda() for x in make_batch(enc, B, D, seed=9)]
    vkw = {"weight": weights("rand", V, 4), "label_smoothing": 0.1}
    nkw = {"weight": weights("rand", L, 5), "label_smoothing": 0.1, "reduction": "sum"}
    results = []
    for graphed in (False, True):
        m = model_from(params, enc, D)
        flat = parallel.attach(m, flat_params=True)
        opt = parallel.FlatAdamax(flat, lr=0.002, max_norm=1.0)
        gs = GraphedTrainStep(m, opt, flat, B, warmup=2, verb_loss_kwargs=vkw, nouns_loss_kwargs=nkw)
        snap = {k: v.detach().clone() for k, v in m.state_dict().items()}

        def restore():
            m.load_state_dict(snap)
            opt.exp_avg.zero_()
            opt.exp_inf.zero_()
            opt.scratch.zero_()

        if graphed:
            gs.capture(batch)
            losses = []
            for _ in range(2):
                restore()
                losses.append(gs(*batch).clone())
        else:
            for dst, src in zip(gs.static_in, batch):
                dst.copy_(src)
            restore()
            losses = [gs._body().clone()]
        torch.cuda.synchronize()
        results.append([x.cpu() for x in losses])
    eager, replays = results
    assert torch.equal(replays[0], replays[1]), replays
    assert torch.allclose(eager[0], replays[0], rtol=1e-5, atol=1e-6), (eager[0], replays[0])
    with pytest.raises(ValueError):
        GraphedTrainStep(m, opt, flat, B, nouns_loss_kwargs={"reduction": "none"})
