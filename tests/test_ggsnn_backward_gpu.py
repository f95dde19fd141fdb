"""-m gpu: the backward of GGSNN.forward (model.ggsnn) on caller-supplied node states and adjacency masks.

The oracle is oracle.ggsnn_forward under torch autograd in fp64 (run on the GPU: at D = 2048 and 768 images the
[B, R, R, D] expansion of the reference is too slow for the CPU), with loss = (out * G).sum() for a random upstream
gradient G.  Tolerance: max|error| <= 3 % of max|reference| per tensor, the bf16 gradient tolerance of the suite."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import situation_recognition_b200 as S
from oracle import ggnn_oracle as O
from situation_recognition_b200.synthetic import make_batch, make_train_json

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GRAD_TOL = 3e-2


def relmax(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def enc_syn():
    return S.imsitu_encoder(make_train_json(seed=0), verbose=False)


@pytest.fixture(scope="module")
def enc_over():
    ann = json.loads(str(np.load(os.path.join(GOLDEN, "encoder_overfitting.npz"))["annotations_json"]))
    return S.imsitu_encoder(ann, verbose=False)


def model_from(params, enc, D, precision="bf16"):
    m = S.FCGGNN(enc, D, backbone=None, precision=precision)
    res = m.load_state_dict({k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in params.items()},
                            strict=False)
    assert not res.unexpected_keys and not res.missing_keys
    return m.cuda().eval()


def oracle_grads(m, hidden, mask, G):
    """fp64 autograd of the oracle GGSNN on the model's weights: (out, d hidden, d mask or None, {param name: grad})."""
    ps = {k: v.detach().double().requires_grad_(True) for k, v in m.ggsnn.named_parameters()}
    h = hidden.detach().cuda().double().requires_grad_(True)
    mk = None if mask is None else mask.detach().cuda().double().requires_grad_(True)
    out = O.ggsnn_forward(ps, h, mask=mk, verb=mask is None)
    (out * G.cuda().double()).sum().backward()
    return out.detach(), h.grad, (None if mk is None else mk.grad), {k: v.grad for k, v in ps.items()}


def cuda_grads(m, hidden, mask, G, mask_grad=True):
    m.zero_grad(set_to_none=True)
    h = hidden.detach().cuda().clone().requires_grad_(True)
    mk = None if mask is None else mask.detach().cuda().clone().requires_grad_(mask_grad)
    out = m.ggsnn(h, mask=mk, verb=mask is None)
    (out * G.cuda()).sum().backward()
    return out.detach(), h.grad, (None if mk is None else mk.grad), {k: p.grad for k, p in m.ggsnn.named_parameters()}


def random_mask(B, R, seed):
    """Asymmetric, real-valued, with self-loops, exact zeros and an all-zero row in every third image."""
    g = torch.Generator().manual_seed(seed)
    mk = torch.rand(B, R, R, generator=g) * 2 - 1
    mk[torch.rand(B, R, R, generator=g) < 0.25] = 0.0
    mk[::3, R // 2, :] = 0.0
    return mk


def case_inputs(name, B, enc_syn, enc_over, D=2048):
    """(model, hidden_state, mask or None) of one oracle case."""
    if name == "golden":
        g = dict(np.load(os.path.join(GOLDEN, "model_overfitting_D256.npz")))
        params = {k[len("param."):]: v for k, v in g.items() if k.startswith("param.")}
        m = model_from(params, enc_over, 256)
        return m, torch.from_numpy(g["ggsnn_in_noun"]), torch.from_numpy(g["ggsnn_mask"])
    R = enc_syn.get_max_role_count()
    m = model_from(O.init_params(504, 190, 2001, D, seed=0), enc_syn, D)
    gen = torch.Generator().manual_seed(B)
    if name == "verb":
        return m, torch.randn(B, D, generator=gen).relu(), None
    hidden = torch.randn(B * R, D, generator=gen).relu()
    if name == "encoder":
        verbs = torch.randint(0, 504, (B,), generator=gen).cuda()
        return m, hidden, m.gather_mask(verbs)[1]
    return m, hidden, random_mask(B, R, seed=B)


@pytest.mark.parametrize("name,B,D", [("golden", None, 256), ("encoder", 11, 2048), ("encoder", 48, 2048),
                                      ("encoder", 768, 2048), ("random", 48, 2048), ("verb", 48, 2048),
                                      ("encoder", 48, 256), ("random", 48, 256)])
def test_ggsnn_gradients_vs_oracle(enc_syn, enc_over, name, B, D):
    """Gradients of hidden_state, mask and all 14 GGSNN tensors.  golden: the reference's own fixture at D = 256 (R = 4);
    encoder: the role-graph mask of random verbs at D = 2048, B = 11 (partial row tiles), 48 and 768 (4 608 rows);
    random: a real-valued asymmetric mask; verb: the verb node.  The D = 256 cases with R = 6 have more mask entries per
    image (36) than the mask-gradient kernel has threads per image (32)."""
    m, hidden, mask = case_inputs(name, B, enc_syn, enc_over, D)
    G = torch.randn(hidden.shape, generator=torch.Generator().manual_seed(7))
    out, dh, dm, dp = cuda_grads(m, hidden, mask, G)
    ref_out, ref_dh, ref_dm, ref_dp = oracle_grads(m, hidden, mask, G)
    errs = {"out": relmax(out, ref_out), "hidden_state": relmax(dh, ref_dh)}
    if mask is not None:
        assert dm.shape == mask.shape and dm.dtype == torch.float32
        errs["mask"] = relmax(dm, ref_dm)
    else:
        assert dm is None
    for k in ref_dp:
        errs[k] = relmax(dp[k], ref_dp[k])
    print("GGSNN_GRADS %s B=%s D=%d %s" % (name, B, D, json.dumps(errs)))
    assert dh.shape == hidden.shape
    for k, e in errs.items():
        assert e <= GRAD_TOL, (k, e)


def test_dropin_composition_matches_oracle(enc_syn):
    """The reference's predict_verb / predict_nouns (model.py:114-168) written out in torch around model.ggsnn: node
    init, F.linear classifiers, losses through verb_loss / nouns_loss.  All 20 trainable tensors get the gradients the
    oracle's autograd gives on the same composition (eval mode, the CUDA path's predicted verbs)."""
    B, D = 16, 256
    R = enc_syn.get_max_role_count()
    params = O.init_params(504, 190, 2001, D, seed=3)
    fv, fn, gt_verb, gt_nouns = make_batch(enc_syn, B, D, seed=8)
    m = model_from(params, enc_syn, D)

    pv = F.linear(m.ggsnn(F.relu(fv.cuda()), verb=True), m.verb_classifier[1].weight, m.verb_classifier[1].bias)
    verbs = pv.argmax(-1)
    role_idx, mask, _ = m.gather_mask(verbs)
    node = F.relu(fn.cuda()[:, None, :] * m.role_emb(role_idx) * m.verb_emb(verbs)[:, None, :]).reshape(B * R, D)
    pn = F.linear(m.ggsnn(node, mask=mask), m.nouns_classifier[1].weight, m.nouns_classifier[1].bias).view(B, R, -1)
    (m.verb_loss(pv, gt_verb.cuda()) + m.nouns_loss(pn, gt_nouns.cuda())).backward()

    t, c = O.build_tables(enc_syn.roles_per_verb, enc_syn.verb_list, enc_syn.role_list)
    _, grads, _ = O.train_step_grads(params, fv, fn, gt_verb, gt_nouns, t, c, 2001, pred_verbs=verbs.cpu())
    names = [k for k, _ in m.named_parameters()]
    assert len(names) == 20
    for k, p in m.named_parameters():
        assert p.grad is not None, k
        assert relmax(p.grad, grads[k]) <= GRAD_TOL, (k, relmax(p.grad, grads[k]))


def test_two_backward_passes_accumulate(enc_syn):
    m, hidden, mask = case_inputs("encoder", 24, enc_syn, None)
    G = torch.randn(hidden.shape, generator=torch.Generator().manual_seed(1)).cuda()
    h = hidden.cuda().requires_grad_(True)
    mk = mask.clone().requires_grad_(True)
    (m.ggsnn(h, mask=mk) * G).sum().backward()
    first = [t.grad.clone() for t in [h, mk] + list(m.ggsnn.parameters())]
    (m.ggsnn(h, mask=mk) * G).sum().backward()
    for t, f in zip([h, mk] + list(m.ggsnn.parameters()), first):
        assert relmax(t.grad, 2 * f) <= 1e-3


def test_flat_buffers_with_fused_paths(enc_syn):
    """One backward over FCGGNN.forward's losses plus a model.ggsnn loss.  With parallel.attach(flat_params=True) every
    path accumulates into the flat .grad views and the chain rule through the folded message weights runs once at the
    end (deferred); without it each call applies its own.  The two differ only in where d/dP is rounded to bf16."""
    from situation_recognition_b200 import parallel
    B, D = 16, 256
    params = O.init_params(504, 190, 2001, D, seed=4)
    fv, fn, gt_verb, gt_nouns = [x.cuda() for x in make_batch(enc_syn, B, D, seed=12)]
    R = enc_syn.get_max_role_count()
    gen = torch.Generator().manual_seed(2)
    hidden = torch.randn(B * R, D, generator=gen).relu().cuda()
    G = (torch.randn(B * R, D, generator=gen) * 1e-2).cuda()

    def run(flat):
        m = model_from(params, enc_syn, D)
        if flat:
            parallel.attach(m, flat_params=True)
        pv, pn, _ = m(fv, gt_verb, img_nouns=fn)
        h = hidden.clone().requires_grad_(True)
        out = m.ggsnn(h, mask=m.gather_mask(gt_verb)[1])
        (m.verb_loss(pv, gt_verb) + m.nouns_loss(pn, gt_nouns) + (out * G).sum()).backward()
        torch.cuda.synchronize()
        return {"hidden_state": h.grad.clone(), **{k: p.grad.clone() for k, p in m.named_parameters()}}

    plain, flat = run(False), run(True)
    for k in plain:
        assert relmax(flat[k], plain[k]) <= 1e-2, (k, relmax(flat[k], plain[k]))


@pytest.mark.parametrize("verb", [False, True])
def test_no_grad_output_is_bit_identical(enc_syn, verb):
    m, hidden, mask = case_inputs("verb" if verb else "encoder", 40, enc_syn, None)
    h = hidden.cuda()
    with torch.no_grad():
        a = m.ggsnn(h, mask=mask, verb=verb)
    b = m.ggsnn(h.clone().requires_grad_(True), mask=mask, verb=verb)
    assert b.requires_grad and not a.requires_grad
    assert torch.equal(a, b.detach())


def test_mask_gradient_only_when_requested(enc_syn, monkeypatch):
    """Without mask.requires_grad the library gets a null dmask (the dot products are skipped) and the mask has no
    gradient; every other gradient is what the run with a mask gradient gives."""
    m, hidden, mask = case_inputs("random", 32, enc_syn, None)
    G = torch.randn(hidden.shape, generator=torch.Generator().manual_seed(3))
    eng = m._engine_for(torch.device("cuda", torch.cuda.current_device()))
    real = eng.lib.srg_ggnn_backward
    seen = []

    def spy(*args):
        seen.append(args[4])
        return real(*args)

    monkeypatch.setattr(eng.lib, "srg_ggnn_backward", spy)
    _, dh0, dm0, dp0 = cuda_grads(m, hidden, mask, G, mask_grad=False)
    dp0 = {k: v.clone() for k, v in dp0.items()}
    _, dh1, dm1, dp1 = cuda_grads(m, hidden, mask, G, mask_grad=True)
    assert seen[0] is None and seen[1] is not None
    assert dm0 is None and dm1 is not None
    assert relmax(dh0, dh1) <= 1e-3
    for k in dp0:
        assert relmax(dp0[k], dp1[k]) <= 1e-3, k


def test_cuda_graph_replay_matches_eager(enc_syn):
    m, hidden, mask = case_inputs("encoder", 24, enc_syn, None)
    G = torch.randn(hidden.shape, generator=torch.Generator().manual_seed(5)).cuda()
    h = hidden.cuda().requires_grad_(True)
    mk = mask.clone().requires_grad_(True)
    leaves = [h, mk] + list(m.ggsnn.parameters())

    def step():
        for t in leaves:
            t.grad = None
        out = m.ggsnn(h, mask=mk)
        (out * G).sum().backward()
        return out

    ref_out = step().detach().clone()
    ref = [t.grad.clone() for t in leaves]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    for t in leaves:
        t.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, ref_out)
    for t, r in zip(leaves, ref):
        assert relmax(t.grad, r) <= 1e-3       # split-K reduce-adds: the sums' order is not fixed


def test_ggnn_backward_argument_checks(enc_syn):
    """srg_ggnn_backward on a live handle and a valid workspace: a bad mode, a null workspace, a null gradient or grads
    struct, a noun-mode call without a mask and a verb-mode call with a dmask return an error code and a message and
    launch nothing."""
    import ctypes
    from situation_recognition_b200 import _lib
    B, D = 4, 256
    R = enc_syn.get_max_role_count()
    m = S.FCGGNN(enc_syn, D, backbone=None).cuda()
    eng = m._engine_for(torch.device("cuda", torch.cuda.current_device()))
    eng.ensure_packed(m, _lib.SRG_PREC_BF16)
    lib, st = eng.lib, eng.stream()
    ws_n = eng.workspace(_lib.SRG_MODE_NOUN, B, _lib.SRG_PREC_BF16, True)
    ws_v = eng.workspace(_lib.SRG_MODE_VERB, B, _lib.SRG_PREC_BF16, True)
    dout = torch.zeros(B * R, D, device="cuda")
    mask = torch.ones(B, R, R, device="cuda")
    dmask = torch.zeros(B, R, R, device="cuda")
    g = _lib.SrgGrads()
    P = _lib.ptr

    def call(mode, dh, mk, dm, grads, ws):
        rc = lib.srg_ggnn_backward(eng.h, mode, P(dh), P(mk), P(dm), None, B, grads, P(ws),
                                   0 if ws is None else ws.numel(), st)
        return rc, (lib.srg_last_error() or b"").decode()

    noun, verb = _lib.SRG_MODE_NOUN, _lib.SRG_MODE_VERB
    for args, msg in [((7, dout, mask, None, ctypes.byref(g), ws_n), "bad mode"),
                      ((noun, dout, mask, None, ctypes.byref(g), None), "null workspace"),
                      ((noun, None, mask, None, ctypes.byref(g), ws_n), "null argument"),
                      ((noun, dout, mask, None, None, ws_n), "null argument"),
                      ((noun, dout, None, dmask, ctypes.byref(g), ws_n), "needs a mask"),
                      ((verb, dout[:B], None, dmask, ctypes.byref(g), ws_v), "dmask must be NULL")]:
        rc, err = call(*args)
        assert rc != 0 and msg in err, (args[0], msg, err)
    torch.cuda.synchronize()


def test_fp32_precision_refuses_a_gradient(enc_syn):
    m = S.FCGGNN(enc_syn, 256, backbone=None, precision="fp32").cuda()
    R = enc_syn.get_max_role_count()
    mask = m.gather_mask(torch.arange(3, device="cuda"))[1]
    with pytest.raises(S._lib.SrgError, match="forward-only"):
        m.ggsnn(torch.rand(3 * R, 256, device="cuda"), mask=mask)            # the parameters require grad
    with pytest.raises(S._lib.SrgError, match="forward-only"):
        m.ggsnn(torch.rand(3, 256, device="cuda", requires_grad=True), verb=True)
    with torch.no_grad():
        out = m.ggsnn(torch.rand(3 * R, 256, device="cuda"), mask=mask)
    assert torch.isfinite(out).all()
