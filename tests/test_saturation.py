"""The value regimes of tests/regimes.py on the fp64 CPU oracle (no GPU needed).

Coverage: every regime is the regime it claims to be, so that a later change of init_params or make_batch fails here
instead of leaving tests/test_saturation_gpu.py silently linear.  Sensitivity: a backward-only bug that takes the
derivative factors of z, r and h_hat clamped to [0.05, 0.95] (h_hat: [-0.95, 0.95]) is invisible at init and moves the
gradients in the saturated regimes by far more than the GPU tests' 3 % tolerance.  Design: the bf16 stash of the CUDA
backward (z and h_hat rounded to bf16, r folded) stays inside that tolerance in every regime."""
import functools

import pytest
import torch

import situation_recognition_b200 as S
from oracle import ggnn_oracle as O
from situation_recognition_b200.synthetic import make_batch, make_train_json
from tests import regimes as G

D, B, R = 256, 48, 6
GRAD_TOL = 3e-2
SATURATED = ("gates_x8", "gate_bias", "fitted")
# gate_bias saturates z and r, not h_hat: only the tensors that take the z / r derivatives are bound to move there
MOVED = {"gates_x8": G.GGSNN_KEYS, "fitted": G.GGSNN_KEYS,
         "gate_bias": tuple("ggsnn.%s.%s" % (k, w) for k in ("W_z", "U_z", "W_r", "U_r") for w in ("weight", "bias"))}


@functools.lru_cache(maxsize=None)
def enc_syn():
    return S.imsitu_encoder(make_train_json(seed=0), verbose=False)


@functools.lru_cache(maxsize=None)
def regime(name):
    """(fp64 params, fp64 batch) of a regime at D = 256, B = 48 (the inputs of the D = 256 GPU cases)."""
    params = O.init_params(504, 190, 2001, D, seed=0)
    p, (fv, fn, gv, gn) = G.REGIMES[name](params, make_batch(enc_syn(), B, D, seed=5), G.tables(enc_syn()))
    return {k: v.double() for k, v in p.items()}, (fv.double(), fn.double(), gv, gn)


@functools.lru_cache(maxsize=None)
def reference(name):
    return G.oracle_step(*regime(name), G.tables(enc_syn()))


def ggsnn_case(mode):
    """model.ggsnn's big_states inputs (as test_saturation_gpu.py builds them) in fp64, with the upstream gradient."""
    params = O.init_params(504, 190, 2001, D, seed=0)
    gen = torch.Generator().manual_seed(17)
    hidden = torch.randn(B * R if mode == "noun" else B, D, generator=gen).relu()
    mask = G.random_mask(B, R, seed=B) if mode == "noun" else None
    params, hidden, mask = G.big_states(params, hidden, mask)
    up = torch.randn(hidden.shape, generator=gen)
    return {k: v.double() for k, v in params.items()}, hidden.double(), mask, up


def assert_saturated(s, h_hat=True):
    for g in ("z", "r"):
        lo, hi = s[g + "_low"], s[g + "_high"]
        assert lo + hi >= 0.3 and lo >= 0.1 and hi >= 0.1, (g, s)
    if h_hat:
        assert s["h_hat_sat"] >= 0.3, s


# ---------------------------------------------------------------------------------------------- coverage
@pytest.mark.parametrize("name", ["init", "gates_x8", "gate_bias", "fitted"])
def test_gate_coverage(name):
    """The gate regimes put >= 30 % of z and of r outside [0.1, 0.9], each tail >= 10 % (and >= 30 % of |h_hat| > 0.9
    where the regime saturates the candidate), on the verb path and on the noun path.  init is linear."""
    trace = G.gate_trace(*regime(name), G.tables(enc_syn()))
    for path, g in trace.items():
        s = G.gate_stats(g)
        if name == "init":
            assert max(s.values()) <= 0.01, (path, s)
        else:
            assert_saturated(s, h_hat=name != "gate_bias")


@pytest.mark.parametrize("mode", ["noun", "verb"])
def test_big_states_coverage(mode):
    params, hidden, mask, _ = ggsnn_case(mode)
    tr = []
    O.ggsnn_forward(O._sub(params, "ggsnn."), hidden, mask=None if mask is None else mask.double(),
                    verb=mask is None, trace=tr)
    assert_saturated(G.gate_stats(G._flat(tr)))


def test_peaked_coverage():
    """Median top-1 softmax probability >= 0.99 on every logit tensor, logit range >= 40, and half of the targets
    are the top-1 while the others sit far down the ranking."""
    _, batch = regime("peaked")
    _, _, (pv, pn, gpn), _ = reference("peaked")
    for x in (pv, pn, gpn):
        assert torch.softmax(x, -1).amax(-1).median() >= 0.99
        assert float(x.max() - x.min()) >= 40
    gt_verb = batch[2]
    hit = pv.argmax(-1) == gt_verb
    assert hit[::2].all() and hit[1::2].float().mean() <= 0.1
    rank = (pv > pv.gather(1, gt_verb[:, None])).sum(-1)
    assert rank[1::2].float().median() >= 10


def test_fitted_coverage():
    (vl, nl, _), _, _, _ = reference("fitted")
    assert float(vl + nl) < 1.0


# ---------------------------------------------------------------------------------------------- sensitivity
def test_clamped_derivative_is_invisible_at_init():
    params, batch = regime("init")
    _, ref, _, _ = reference("init")
    with G.derivative("clamped"):
        _, got, _, _ = G.oracle_step(params, batch, G.tables(enc_syn()))
    for k in ref:
        assert G.relmax(got[k], ref[k]) <= 1e-12, k


@pytest.mark.parametrize("name", SATURATED)
def test_clamped_derivative_moves_saturated_gradients(name):
    params, batch = regime(name)
    _, ref, _, _ = reference(name)
    with G.derivative("clamped"):
        _, got, _, _ = G.oracle_step(params, batch, G.tables(enc_syn()))
    for k in MOVED[name]:
        assert G.relmax(got[k], ref[k]) >= 3 * GRAD_TOL, (k, G.relmax(got[k], ref[k]))


@pytest.mark.parametrize("mode", ["noun", "verb"])
def test_clamped_derivative_moves_big_states_gradients(mode):
    params, hidden, mask, up = ggsnn_case(mode)
    _, dh, dm, ref = G.oracle_ggsnn(params, hidden, mask, up)
    with G.derivative("clamped"):
        _, gdh, gdm, got = G.oracle_ggsnn(params, hidden, mask, up)
    errs = {k: G.relmax(got[k], ref[k]) for k in ref}
    errs["hidden_state"] = G.relmax(gdh, dh)
    if mask is not None:
        errs["mask"] = G.relmax(gdm, dm)
    for k, e in errs.items():
        assert e >= 3 * GRAD_TOL, (k, e)


# ---------------------------------------------------------------------------------------------- designed rounding
@pytest.mark.parametrize("name", ["init", "gates_x8", "gate_bias", "peaked", "fitted"])
def test_bf16_stash_rounding_within_tolerance(name):
    """The derivative factors rebuilt from the bf16 stash (z, h_hat rounded; r folded to min(r, 1 - r) first, as
    gate_fold in gemm.cuh) alone move no gradient by more than half of the 3 % tolerance, leaving the rest to the
    bf16 GEMM operands.  With r stashed unfolded, the r-gate gradients of gate_bias and fitted exceed 3 % by
    themselves."""
    params, batch = regime(name)
    _, ref, _, _ = reference(name)
    with G.derivative("bf16_stash"):
        _, got, _, _ = G.oracle_step(params, batch, G.tables(enc_syn()))
    for k in ref:
        assert G.relmax(got[k], ref[k]) <= GRAD_TOL / 2, (k, G.relmax(got[k], ref[k]))
