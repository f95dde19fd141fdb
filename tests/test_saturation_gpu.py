"""-m gpu: the CUDA paths where the GRU gates saturate and the logits are peaked (tests/regimes.py), against fp64 autograd
of the oracle.

The rest of the GPU suite runs at the reference's default init, where z and r stay near 0.5 and the logits span about
+-1: there the backward's derivative factors z (1 - z), 1 - z, r (1 - r) and 1 - h_hat^2, rebuilt from the bf16 stash,
and the loss kernels' rescaled softmax statistics have no visible effect.  Here every case runs in a regime whose
coverage tests/test_saturation.py asserts on the CPU, with the suite's own bounds (logits <= 2e-2 and every gradient
tensor <= 3e-2 of max|reference|, losses within 2e-3 relative; 1e-4 for the fp32-parity forward) or, where the
designed bf16 rounding alone exceeds them, twice what a bf16 emulation of that rounding gives (see EMUL_FACTOR).  Each case prints a
`PARITY {json}` line with the max-relative and relative-Frobenius error per tensor.  The oracle runs on the CPU at
D = 256 and on the GPU (still fp64) at D = 2048."""
import functools
import json

import pytest
import torch
import torch.nn.functional as F

import situation_recognition_b200 as S
from oracle import ggnn_oracle as O
from situation_recognition_b200.synthetic import make_batch, make_train_json
from tests import regimes as G

pytestmark = pytest.mark.gpu

LOGIT_TOL, GRAD_TOL, LOSS_TOL, FP32_TOL = 2e-2, 3e-2, 2e-3, 1e-4
R = 6


@functools.lru_cache(maxsize=None)
def enc_syn():
    return S.imsitu_encoder(make_train_json(seed=0), verbose=False)


def oracle_device(D):
    return "cuda" if D >= 2048 else "cpu"


@functools.lru_cache(maxsize=None)
def regime_inputs(name, D, B):
    """(params, batch) of a regime on the CPU; built on the oracle's device (fitting at D = 2048 runs on the GPU)."""
    dev = oracle_device(D)
    params = {k: v.to(dev) for k, v in O.init_params(504, 190, 2001, D, seed=0).items()}
    batch = tuple(x.to(dev) for x in make_batch(enc_syn(), B, D, seed=5))
    p, b = G.REGIMES[name](params, batch, G.tables(enc_syn()))
    return {k: v.cpu() for k, v in p.items()}, tuple(x.cpu() for x in b)


def model_from(params, D, precision="bf16"):
    m = S.FCGGNN(enc_syn(), D, backbone=None, precision=precision)
    res = m.load_state_dict(params, strict=False)
    assert not res.unexpected_keys and not res.missing_keys
    return m.cuda().eval()


def errors(got, ref):
    return {"max_rel": G.relmax(got, ref), "rel_fro": G.relfro(got, ref)}


def report(name, **values):
    print("PARITY " + json.dumps({"test": name, **values}))


def keep_masks(B, D, seed=5):
    g = torch.Generator().manual_seed(seed)
    return tuple(torch.rand(n, D, generator=g) < 0.5 for n in (B, B * R, B * R))


# ---------------------------------------------------------------------------------------------- bounds
# Each check compares with fp64.  Its bound is the suite's own tolerance, or, where the designed rounding alone is
# larger, EMUL_FACTOR times the largest error of the bf16 emulation (regimes.bf16_emulation: bf16 GEMM operands in the
# forward and in both backward GEMMs, derivative factors from the bf16 stash) in the same group of tensors and regime.
# The CUDA path rounds at other places (folded gate weights, summation order, tanh.approx), so its error is another
# draw of the same size, not the same number; a factor of 2 admits that and fails a defect that adds as much again.
EMUL_FACTOR = 2.0


def emulated_bound(tol, emul_errs):
    return max(tol, EMUL_FACTOR * max(emul_errs))


def check(group, tol, errs, emul):
    """errs / emul: {tensor: error against fp64} of the CUDA path and of the emulation."""
    bound = emulated_bound(tol, emul.values())
    for k, e in errs.items():
        assert e["max_rel"] <= bound, (group, k, e, "bound %.4g" % bound)


# ---------------------------------------------------------------------------------------------- training step
STEP_CASES = [("init", 256, 48, "eval"), ("gates_x8", 256, 48, "eval"), ("gate_bias", 256, 48, "eval"),
              ("peaked", 256, 48, "eval"), ("fitted", 256, 48, "eval"),
              ("gates_x8", 2048, 16, "eval"), ("fitted", 2048, 16, "eval"),
              ("gates_x8", 256, 48, "one_row_per_slot"), ("gate_bias", 256, 48, "cta_group_1"),
              ("gates_x8", 256, 48, "train_keeps"), ("fitted", 256, 48, "flat")]


@pytest.mark.parametrize("regime,D,B,variant", STEP_CASES)
def test_training_step_vs_oracle(regime, D, B, variant):
    """verb_loss + nouns_loss backward (sr.py's step), the oracle's predicted-verb path conditioned on the CUDA path's
    own argmax: the three logits, the three losses, all 20 gradients and dL/dfeat of both paths.  Variants: the
    reference's one row per role slot instead of compact rows, cta_group 1, training mode with explicit dropout keep
    masks, and flat gradient buffers with the deferred chain rule."""
    params, (fv, fn, gt_verb, gt_nouns) = regime_inputs(regime, D, B)
    m = model_from(params, D)
    eng = m._engine_for(torch.device("cuda", 0))
    keeps = (None, None, None)
    if variant == "one_row_per_slot":
        eng.set_compact_rows(False)
    elif variant == "cta_group_1":
        eng.set_cta_group(1)
    elif variant == "train_keeps":
        keeps = keep_masks(B, D)
        m.train()
        m.dropout_masks = tuple(k.to(torch.uint8).cuda() for k in keeps)
    elif variant == "flat":
        from situation_recognition_b200 import parallel
        parallel.attach(m, flat_params=True)
    xv = fv.cuda().requires_grad_(True)
    xn = fn.cuda().requires_grad_(True)
    gv, gn = gt_verb.cuda(), gt_nouns.cuda()
    mpv, mpn, mgpn = m(xv, gv, img_nouns=xn)
    lv, ln, lg = m.verb_loss(mpv, gv), m.nouns_loss(mpn, gn), m.nouns_loss(mgpn, gn)
    (lv + ln).backward()
    pred = mpv.argmax(-1).cpu()
    args = (params, (fv, fn, gt_verb, gt_nouns), G.tables(enc_syn()), pred, keeps, True)
    (vl, nl, gl), ref, (pv, pn, gpn), (dfv, dfn) = G.oracle_step(*args, device=oracle_device(D))
    with G.bf16_emulation():
        (evl, enl, egl), eref, (epv, epn, egpn), (edfv, edfn) = G.oracle_step(*args, device=oracle_device(D))
    if regime == "fitted":
        assert float(vl + nl) < 1.0, "not a fitted point: loss %.3f" % float(vl + nl)
    grads = {k: errors(p.grad if p.grad is not None else torch.zeros_like(p), ref[k]) for k, p in m.named_parameters()}
    logits = {"verb": errors(mpv, pv), "pred_nouns": errors(mpn, pn), "gt_nouns": errors(mgpn, gpn)}
    feats = {"feat_v": errors(xv.grad, dfv), "feat_n": errors(xn.grad, dfn)}
    losses = {"cuda": [lv.item(), ln.item(), lg.item()], "oracle": [float(vl), float(nl), float(gl)],
              "emulated": [float(evl), float(enl), float(egl)]}
    emul = {"logits": {k: G.relmax(a, b) for k, a, b in zip(logits, (epv, epn, egpn), (pv, pn, gpn))},
            "grads": {k: G.relmax(eref[k], ref[k]) for k in ref},
            "feat_grads": {"feat_v": G.relmax(edfv, dfv), "feat_n": G.relmax(edfn, dfn)},
            "losses": {i: abs(e - o) / abs(o) for i, (e, o) in enumerate(zip(losses["emulated"], losses["oracle"]))}}
    report("saturation_training_step[%s,D=%d,B=%d,%s]" % (regime, D, B, variant), logits=logits, losses=losses,
           grads=grads, feat_grads=feats, emulated_max_rel=emul)
    check("logits", LOGIT_TOL, logits, emul["logits"])
    check("grads", GRAD_TOL, grads, emul["grads"])
    check("feat_grads", GRAD_TOL, feats, emul["feat_grads"])
    loss_bound = emulated_bound(LOSS_TOL, emul["losses"].values())
    for mine, want in zip(losses["cuda"], losses["oracle"]):
        assert abs(mine - want) <= loss_bound * abs(want), (losses, loss_bound)


# ---------------------------------------------------------------------------------------------- model.ggsnn
@pytest.mark.parametrize("regime", ["big_states", "gates_x8"])
@pytest.mark.parametrize("mode", ["noun", "verb"])
def test_ggsnn_vs_oracle(regime, mode):
    """GGSNN.forward on caller-supplied states (and, in noun mode, a random real-valued mask that requires grad):
    the output, d hidden, d mask and the 14 GGSNN gradients for loss = (out * G).sum()."""
    D, B = 256, 48
    params = O.init_params(504, 190, 2001, D, seed=0)
    gen = torch.Generator().manual_seed(17)
    hidden = torch.randn(B * R if mode == "noun" else B, D, generator=gen).relu()
    mask = G.random_mask(B, R, seed=B) if mode == "noun" else None
    if regime == "big_states":
        params, hidden, mask = G.big_states(params, hidden, mask)
    else:
        params, _ = G.gates_x8(params, None, None)
    up = torch.randn(hidden.shape, generator=gen)
    m = model_from(params, D)
    h = hidden.cuda().requires_grad_(True)
    mk = None if mask is None else mask.cuda().requires_grad_(True)
    out = m.ggsnn(h, mask=mk, verb=mask is None)
    (out * up.cuda()).sum().backward()
    refs = G.oracle_ggsnn(params, hidden, mask, up)
    with G.bf16_emulation():
        emuls = G.oracle_ggsnn(params, hidden, mask, up)

    def named(res):
        o, dh, dm, dp = res
        return {"out": o, "hidden_state": dh, **({} if dm is None else {"mask": dm}), **dp}

    got = named((out, h.grad, None if mk is None else mk.grad, {k: p.grad for k, p in m.ggsnn.named_parameters()}))
    ref, emu = named(refs), named(emuls)
    errs = {k: errors(got[k], ref[k]) for k in ref}
    emul = {k: G.relmax(emu[k], ref[k]) for k in ref}
    report("saturation_ggsnn[%s,%s]" % (regime, mode), errors=errs, emulated_max_rel=emul)
    check("out", LOGIT_TOL, {"out": errs["out"]}, {"out": emul["out"]})
    check("grads", GRAD_TOL, {k: e for k, e in errs.items() if k != "out"},
          {k: e for k, e in emul.items() if k != "out"})


# ---------------------------------------------------------------------------------------------- loss kernels
@pytest.mark.parametrize("route", ["softmax_stats", "three_pass"])
def test_loss_kernels_at_peaked(route):
    """verb_loss / nouns_loss and their d(loss)/d(logits) on the CUDA path's own peaked logits against F.cross_entropy
    in fp64 on the same logits: <= 1e-5 relative on the loss, <= 1e-4 of max on dlogits.  softmax_stats: the very
    tensors predict_* returned, so the loss kernels use the classifier's per-tile row max / sum-exp; three_pass: a
    clone, which they read three times instead.  Separates the statistics' rescaling from GEMM rounding."""
    D, B = 256, 48
    params, (fv, fn, gt_verb, gt_nouns) = regime_inputs("peaked", D, B)
    m = model_from(params, D)
    gv, gn = gt_verb.cuda(), gt_nouns.cuda()
    with torch.no_grad():
        outs = m(fv.cuda(), gv, img_nouns=fn.cuda())
    errs = {}
    for name, logits in zip(("verb", "pred_nouns", "gt_nouns"), outs):
        x = logits if route == "softmax_stats" else logits.clone()
        assert (getattr(x, "_srg_stats", None) is not None) == (route == "softmax_stats")
        x.requires_grad_(True)
        loss = m.verb_loss(x, gv) if name == "verb" else m.nouns_loss(x, gn)
        loss.backward()
        ref_x = logits.detach().double().cpu().requires_grad_(True)
        ref = F.cross_entropy(ref_x, gt_verb) if name == "verb" else O.nouns_loss(ref_x, gt_nouns, 2001)
        ref.backward()
        errs[name] = {"loss": abs(loss.item() - ref.item()) / abs(ref.item()), "dlogits": errors(x.grad, ref_x.grad),
                      "logit_range": float(logits.max() - logits.min())}
    report("saturation_loss_kernels[peaked,%s]" % route, errors=errs)
    for k, e in errs.items():
        assert e["loss"] <= 1e-5, (k, e)
        assert e["dlogits"]["max_rel"] <= 1e-4, (k, e)


# ---------------------------------------------------------------------------------------------- fp32-parity forward
@pytest.mark.parametrize("regime", ["gates_x8", "peaked"])
def test_fp32_forward_vs_oracle(regime):
    """precision="fp32": logits <= 1e-4 of max|logit| against fp64, and the same argmax on every row whose fp64
    top-1 / top-2 margin exceeds 1e-3 of the tensor's logit range (at the error bound no such row can flip)."""
    D, B = 256, 48
    params, (fv, fn, gt_verb, _) = regime_inputs(regime, D, B)
    m = model_from(params, D, precision="fp32")
    with torch.no_grad():
        outs = m(fv.cuda(), gt_verb.cuda(), img_nouns=fn.cuda())
    p64 = {k: v.double() for k, v in params.items()}
    with torch.no_grad():
        refs = O.forward(p64, fv.double(), fn.double(), gt_verb, *G.tables(enc_syn()),
                         pred_verbs=outs[0].argmax(-1).cpu())
    res = {}
    for name, got, ref in zip(("verb", "pred_nouns", "gt_nouns"), outs, refs):
        got, ref = got.cpu().reshape(-1, ref.shape[-1]), ref.reshape(-1, ref.shape[-1])
        top2 = ref.topk(2, -1).values
        clear = (top2[:, 0] - top2[:, 1]) > 1e-3 * float(ref.max() - ref.min())
        res[name] = {**errors(got, ref), "clear_rows": int(clear.sum()), "rows": int(clear.numel()),
                     "argmax_flips": int((got.argmax(-1) != ref.argmax(-1))[clear].sum())}
    report("saturation_fp32_forward[%s]" % regime, errors=res)
    for k, e in res.items():
        assert e["max_rel"] <= FP32_TOL, (k, e)
        assert e["clear_rows"] > 0 and e["argmax_flips"] == 0, (k, e)
