"""-m gpu: gradients w.r.t. the backbone features (dL/dfeat) of the fused verb and noun paths.

The reference is the oracle under torch autograd in fp64 with the feature tensors as leaves, run on the GPU (at D = 2048
and 768 images the [B, R, R, D] expansion of the reference is too slow for the CPU).  `oracle_nouns` below is
oracle.predict_nouns with its role ids and mask moved to the features' device.  Tolerance: max|error| <= 3 % of
max|reference|, the bf16 gradient tolerance of the suite."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import situation_recognition_b200 as S
from oracle import ggnn_oracle as O
from situation_recognition_b200 import _lib, parallel
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


def tables(enc):
    return O.build_tables(enc.roles_per_verb, enc.verb_list, enc.role_list)


def model_from(params, enc, D):
    m = S.FCGGNN(enc, D, backbone=None)
    res = m.load_state_dict({k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in params.items()},
                            strict=False)
    assert not res.unexpected_keys and not res.missing_keys
    return m.cuda().eval()


def case_model(name, enc_syn, enc_over):
    """(model, encoder): the overfitting encoder's golden weights at D = 256 (R = 4), or synthetic-504 at D = 2048."""
    if name == "over":
        g = dict(np.load(os.path.join(GOLDEN, "model_overfitting_D256.npz")))
        return model_from({k[len("param."):]: v for k, v in g.items() if k.startswith("param.")}, enc_over, 256), enc_over
    return model_from(O.init_params(504, 190, 2001, 2048, seed=0), enc_syn, 2048), enc_syn


def p64(m):
    return {k: v.detach().double() for k, v in m.named_parameters()}


def oracle_nouns(p, feat, verbs, t, c, keep=None):
    """oracle.predict_nouns (model.py:114-155) on the features' device."""
    B, R = feat.shape[0], t.shape[1]
    v = verbs.cpu().numpy()
    role_idx = torch.from_numpy(O.get_role_ids_batch(t, v)).to(feat.device)
    ve = p["verb_emb.weight"][verbs.to(feat.device)]
    node = F.relu(feat[:, None, :] * p["role_emb.weight"][role_idx] * ve[:, None, :]).reshape(B * R, -1)
    mask = torch.from_numpy(O.get_adj_matrix_noself(c, v, R)).to(feat.device, feat.dtype)
    out = O.ggsnn_forward(O._sub(p, "ggsnn."), node, mask=mask)
    logits = O.linear(O.dropout(out, keep, 0.5), p["nouns_classifier.1.weight"], p["nouns_classifier.1.bias"])
    return logits.view(B, R, -1)


def leaf(x, dtype=torch.float32):
    return x.detach().cuda().to(dtype).clone().requires_grad_(True)


def signed_feats(B, D, seed):
    """Signed features with exact zeros (the node ReLUs see both signs)."""
    g = torch.Generator().manual_seed(seed)
    f = torch.randn(B, D, generator=g)
    f[torch.rand(B, D, generator=g) < 0.1] = 0.0
    return f


def path_grads(m, enc, B, compact=True, seed=3):
    """dL/dfeat of predict_verb and predict_nouns (eval mode) for loss = (logits * G).sum(), with the oracle's."""
    D = m.D
    m._engine_for(torch.device("cuda", 0)).set_compact_rows(compact)
    g = torch.Generator().manual_seed(seed)
    fv, fn = signed_feats(B, D, seed), signed_feats(B, D, seed + 1)
    verbs = torch.randint(0, enc.get_num_verbs(), (B,), generator=g)
    Gv = torch.randn(B, enc.get_num_verbs(), generator=g)
    Gn = torch.randn(B, enc.get_max_role_count(), enc.get_num_labels(), generator=g)
    xv, xn = leaf(fv), leaf(fn)
    (m.predict_verb(xv, B) * Gv.cuda()).sum().backward()
    (m.predict_nouns(xn, verbs.cuda(), B) * Gn.cuda()).sum().backward()
    p = p64(m)
    t, c = tables(enc)
    ov, on = leaf(fv, torch.float64), leaf(fn, torch.float64)
    (O.predict_verb(p, ov) * Gv.cuda().double()).sum().backward()
    (oracle_nouns(p, on, verbs, t, c) * Gn.cuda().double()).sum().backward()
    return (xv.grad, xn.grad), (ov.grad, on.grad)


@pytest.mark.parametrize("compact", [True, False])
@pytest.mark.parametrize("name,B", [("over", 16), ("syn", 11), ("syn", 48), ("syn", 768)])
def test_feature_gradients_vs_oracle(enc_syn, enc_over, name, B, compact):
    """predict_verb and predict_nouns: dL/dfeat against fp64 autograd of the oracle, on both row layouts."""
    m, enc = case_model(name, enc_syn, enc_over)
    (gv, gn), (rv, rn) = path_grads(m, enc, B, compact)
    assert gv.shape == (B, m.D) and gv.dtype == torch.float32 and gn.shape == (B, m.D)
    errs = {"verb": relmax(gv, rv), "nouns": relmax(gn, rn)}
    print("FEAT_GRADS %s B=%d compact=%s %s" % (name, B, compact, json.dumps(errs)))
    for k, e in errs.items():
        assert e <= GRAD_TOL, (k, e)


def test_row_layouts_agree(enc_syn):
    m, enc = case_model("syn", enc_syn, None)
    (a_v, a_n), _ = path_grads(m, enc, 48, compact=True)
    (b_v, b_n), _ = path_grads(m, enc, 48, compact=False)
    assert relmax(a_v, b_v) <= 1e-3 and relmax(a_n, b_n) <= 1e-3


def _train_step(m, fv, fn, gt_verb, gt_nouns):
    torch.manual_seed(123)        # the model draws its first Philox seed from torch's CPU generator
    m.zero_grad(set_to_none=True)
    pv, pn, gpn = m.forward_features(fv, fn, gt_verb)
    (m.verb_loss(pv, gt_verb) + m.nouns_loss(pn, gt_nouns)).backward()
    return pv, m.last_drop_seed


@pytest.mark.parametrize("B", [48, 768])
def test_training_step_feature_gradients(enc_syn, B):
    """forward_features in train mode (Philox dropout, replayed through model.dropout_mask) with the launcher's loss:
    dL/dfeat_v and dL/dfeat_n against the oracle (its predicted-verb path under the CUDA argmax); the 20 parameter
    gradients agree with a run whose features need no gradient."""
    D, R = 2048, enc_syn.get_max_role_count()
    params = O.init_params(504, 190, 2001, D, seed=0)
    fv, fn, gt_verb, gt_nouns = [x.cuda() for x in make_batch(enc_syn, B, D, seed=41)]
    fv, fn = fv - 0.4, fn - 0.4                      # both signs at the verb node's ReLU
    m = model_from(params, enc_syn, D).train()
    xv, xn = leaf(fv), leaf(fn)
    pv, seed = _train_step(m, xv, xn, gt_verb, gt_nouns)
    with_feat = {k: p.grad.clone() for k, p in m.named_parameters()}
    masks = [m.dropout_mask(w, r, seed) for w, r in ((0, B), (1, B * R), (2, B * R))]
    m2 = model_from(params, enc_syn, D).train()
    _, seed2 = _train_step(m2, fv, fn, gt_verb, gt_nouns)
    assert torch.equal(seed, seed2)
    for k, p in m2.named_parameters():
        assert relmax(with_feat[k], p.grad) <= 1e-3, k
    p = p64(m)
    t, c = tables(enc_syn)
    ov, on = leaf(fv, torch.float64), leaf(fn, torch.float64)
    opv = O.predict_verb(p, ov, masks[0])
    opn = oracle_nouns(p, on, pv.argmax(-1), t, c, masks[1])
    (O.verb_loss(opv, gt_verb) + O.nouns_loss(opn, gt_nouns, 2001)).backward()
    errs = {"feat_v": relmax(xv.grad, ov.grad), "feat_n": relmax(xn.grad, on.grad)}
    print("TRAIN_FEAT_GRADS B=%d %s" % (B, json.dumps(errs)))
    for k, e in errs.items():
        assert e <= GRAD_TOL, (k, e)


def _all_losses(m, outs, gt_verb, gt_nouns):
    pv, pn, gpn = outs
    return m.verb_loss(pv, gt_verb) + m.nouns_loss(pn, gt_nouns) + m.nouns_loss(gpn, gt_nouns)


def test_shared_input_gradient_is_the_sum(enc_syn):
    """forward_features(f, f) and forward(img) without a backbone: one tensor feeds the verb path and both noun paths."""
    B, D = 48, 2048
    m = model_from(O.init_params(504, 190, 2001, D, seed=0), enc_syn, D)
    f, _, gt_verb, gt_nouns = [x.cuda() for x in make_batch(enc_syn, B, D, seed=43)]
    f = f - 0.4
    x = leaf(f)
    outs = m.forward_features(x, x, gt_verb)
    _all_losses(m, outs, gt_verb, gt_nouns).backward()
    img = leaf(f)
    _all_losses(m, m(img, gt_verb), gt_verb, gt_nouns).backward()
    assert relmax(img.grad, x.grad) <= 1e-6
    p = p64(m)
    t, c = tables(enc_syn)
    o = leaf(f, torch.float64)
    opv, opn, ogn = O.predict_verb(p, o), oracle_nouns(p, o, outs[0].argmax(-1), t, c), oracle_nouns(p, o, gt_verb, t, c)
    (O.verb_loss(opv, gt_verb) + O.nouns_loss(opn, gt_nouns, 2001) + O.nouns_loss(ogn, gt_nouns, 2001)).backward()
    assert relmax(x.grad, o.grad) <= GRAD_TOL, relmax(x.grad, o.grad)


def test_trainable_adapter_weight_gradient(enc_over):
    """A trainable nn.Linear in front of both inputs of forward_features: its weight gradient is the oracle's."""
    B, D = 16, 256
    g = dict(np.load(os.path.join(GOLDEN, "model_overfitting_D256.npz")))
    m = model_from({k[len("param."):]: v for k, v in g.items() if k.startswith("param.")}, enc_over, D)
    gen = torch.Generator().manual_seed(5)
    xv, xn = torch.randn(B, D, generator=gen).cuda(), torch.randn(B, D, generator=gen).cuda()
    gt_verb = torch.randint(0, enc_over.get_num_verbs(), (B,), generator=gen).cuda()
    gt_nouns = torch.randint(0, enc_over.get_num_labels(), (B, 3, enc_over.get_max_role_count()), generator=gen).cuda()
    lin = torch.nn.Linear(D, D).cuda()
    outs = m.forward_features(lin(xv), lin(xn), gt_verb)
    L = enc_over.get_num_labels()
    _all_losses(m, outs, gt_verb, gt_nouns).backward()
    p = p64(m)
    t, c = tables(enc_over)
    W, b = leaf(lin.weight, torch.float64), leaf(lin.bias, torch.float64)
    fv, fn = O.linear(xv.double(), W, b), O.linear(xn.double(), W, b)
    opv, opn, ogn = O.predict_verb(p, fv), oracle_nouns(p, fn, outs[0].argmax(-1), t, c), oracle_nouns(p, fn, gt_verb, t, c)
    (O.verb_loss(opv, gt_verb) + O.nouns_loss(opn, gt_nouns, L) + O.nouns_loss(ogn, gt_nouns, L)).backward()
    errs = {"weight": relmax(lin.weight.grad, W.grad), "bias": relmax(lin.bias.grad, b.grad)}
    print("ADAPTER_GRADS %s" % json.dumps(errs))
    for k, e in errs.items():
        assert e <= GRAD_TOL, (k, e)


def test_bf16_features_get_the_cast_fp32_gradient(enc_syn):
    B, D = 48, 2048
    m = model_from(O.init_params(504, 190, 2001, D, seed=0), enc_syn, D)
    f = signed_feats(B, D, 9).cuda().bfloat16()
    verbs = torch.randint(0, 504, (B,), generator=torch.Generator().manual_seed(2)).cuda()
    for run in (lambda x: m.predict_verb(x, B), lambda x: m.predict_nouns(x, verbs, B)):
        x32, xbf = leaf(f.float()), leaf(f, torch.bfloat16)
        run(x32).square().sum().backward()
        run(xbf).square().sum().backward()
        assert xbf.grad.dtype == torch.bfloat16 and torch.equal(xbf.grad, x32.grad.bfloat16())


def test_inactive_nodes_give_exact_zeros(enc_syn):
    """dL/dfeat is exactly 0 wherever the node's ReLU is inactive: feat <= 0 on the verb node; on the role graph, columns
    where every real role node of the image is <= 0 (feat = 0 among them)."""
    B, D = 48, 2048
    m = model_from(O.init_params(504, 190, 2001, D, seed=0), enc_syn, D)
    f = signed_feats(B, D, 11).cuda()
    verbs = torch.randint(0, 504, (B,), generator=torch.Generator().manual_seed(4)).cuda()
    xv, xn = leaf(f), leaf(f)
    m.predict_verb(xv, B).square().sum().backward()
    m.predict_nouns(xn, verbs, B).square().sum().backward()
    assert (xv.grad[f <= 0] == 0).all() and (xv.grad[f > 0] != 0).float().mean() > 0.9
    t, c = tables(enc_syn)
    role_idx = torch.from_numpy(O.get_role_ids_batch(t, verbs.cpu().numpy())).cuda()
    with torch.no_grad():
        node = F.relu((f[:, None, :] * m.role_emb.weight[role_idx]) * m.verb_emb.weight[verbs][:, None, :])
    inactive = (node == 0).all(1)
    assert inactive.float().mean() > 0.05 and (f == 0).float().mean() > 0.05
    assert (xn.grad[inactive] == 0).all() and (xn.grad[~inactive] != 0).float().mean() > 0.9


def _feature_grads(m, fv, fn, gt_verb, gt_nouns):
    xv, xn = leaf(fv), leaf(fn)
    _all_losses(m, m.forward_features(xv, xn, gt_verb), gt_verb, gt_nouns).backward()
    return xv.grad, xn.grad


def test_feature_gradients_are_deterministic_and_equal_in_flat_mode(enc_syn):
    """Two identical backward passes give bit-identical dL/dfeat (no atomics in the feature reduction; only the weight
    gradient GEMMs are split-K), and the flat-buffer mode with the deferred chain rule gives the same bits."""
    B, D = 48, 2048
    params = O.init_params(504, 190, 2001, D, seed=0)
    fv, fn, gt_verb, gt_nouns = [x.cuda() for x in make_batch(enc_syn, B, D, seed=45)]
    fv = fv - 0.4
    m = model_from(params, enc_syn, D)
    a = _feature_grads(m, fv, fn, gt_verb, gt_nouns)
    b = _feature_grads(m, fv, fn, gt_verb, gt_nouns)
    mf = model_from(params, enc_syn, D)
    flat = parallel.attach(mf, flat_params=True)
    flat.zero()
    c = _feature_grads(mf, fv, fn, gt_verb, gt_nouns)
    torch.cuda.synchronize()
    for x, y, z in zip(a, b, c):
        assert torch.equal(x, y) and torch.equal(x, z)
    assert mf.ggsnn.W_p.weight.grad.abs().max() > 0


def test_cuda_graph_replay_matches_eager(enc_syn):
    B, D = 48, 2048
    m = model_from(O.init_params(504, 190, 2001, D, seed=0), enc_syn, D)
    fv, fn, gt_verb, gt_nouns = [x.cuda() for x in make_batch(enc_syn, B, D, seed=47)]
    fv = fv - 0.4
    eager = _feature_grads(m, fv, fn, gt_verb, gt_nouns)
    xv, xn = leaf(fv), leaf(fn)

    def step():
        _all_losses(m, m.forward_features(xv, xn, gt_verb), gt_verb, gt_nouns).backward()

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    m.zero_grad(set_to_none=True)
    xv.grad = xn.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(xv.grad, eager[0]) and torch.equal(xn.grad, eager[1])


def test_feature_gradient_only_on_request(enc_syn, monkeypatch):
    """The stages pass dfeat = NULL unless a feature requires grad, and the logits do not depend on it."""
    B, D = 24, 2048
    m = model_from(O.init_params(504, 190, 2001, D, seed=0), enc_syn, D)
    fv, fn, gt_verb, gt_nouns = [x.cuda() for x in make_batch(enc_syn, B, D, seed=49)]
    lib = m._engine_for(fv.device).lib
    seen = []
    for name, arg in (("srg_nouns_backward_feat", 14), ("srg_verb_backward_feat", 10)):
        orig = getattr(lib, name)

        def spy(*a, _orig=orig, _name=name, _arg=arg):
            seen.append((_name, a[_arg] is not None))
            return _orig(*a)
        monkeypatch.setattr(lib, name, spy)
    outs = []
    for want in (False, True):
        seen.clear()
        xv, xn = (leaf(fv), leaf(fn)) if want else (fv, fn)
        o = m.forward_features(xv, xn, gt_verb)
        _all_losses(m, o, gt_verb, gt_nouns).backward()
        torch.cuda.synchronize()
        assert sorted(seen) == sorted([("srg_verb_backward_feat", want)] + [("srg_nouns_backward_feat", want)] * 2)
        outs.append([t.detach().clone() for t in o])
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_fp32_precision_refuses_feature_gradients(enc_syn):
    m = model_from(O.init_params(504, 190, 2001, 256, seed=0), enc_syn, 256)
    m.precision = "fp32"
    m.requires_grad_(False)               # only the features ask for a gradient
    x = leaf(torch.rand(4, 256))
    with pytest.raises(_lib.SrgError, match="forward-only"):
        m.predict_verb(x, 4)
    with pytest.raises(_lib.SrgError, match="forward-only"):
        m.predict_nouns(x, torch.zeros(4, dtype=torch.long, device="cuda"), 4)


def test_entry_points_refuse_bad_arguments_on_a_live_handle(enc_syn):
    """Null workspace, null grads struct, fp32-packed weights: an error code and a message, and nothing launched or
    written."""
    B, D = 4, 256
    m = model_from(O.init_params(504, 190, 2001, D, seed=0), enc_syn, D)
    eng = m._engine_for(torch.device("cuda", 0))
    feat = torch.rand(B, D, device="cuda")
    verb = torch.zeros(B, dtype=torch.long, device="cuda")
    grads = {n: torch.zeros_like(p) for n, p in zip(_lib._PARAM_FIELDS + ["role_emb", "verb_emb"],
                                                    eng.param_list(m) + [m.role_emb.weight, m.verb_emb.weight])}
    sg = _lib.SrgGrads(**{n: ctypes.c_void_p(t.data_ptr()) for n, t in grads.items()})
    dfeat = torch.zeros(B, D, device="cuda")
    ptr = _lib.ptr

    def call(mode, ws, g):
        wp, wn = (ptr(ws), ws.numel()) if ws is not None else (None, 0)
        if mode == _lib.SRG_MODE_NOUN:
            return eng.lib.srg_nouns_backward_feat(eng.h, None, 0, 1, ptr(feat), ptr(verb), B, ptr(m.role_emb.weight),
                                                   ptr(m.verb_emb.weight), None, 0.0, None, 0, g, ptr(dfeat), wp, wn,
                                                   eng.stream())
        return eng.lib.srg_verb_backward_feat(eng.h, None, 0, 1, B, None, 0.0, None, 0, g, ptr(dfeat), wp, wn,
                                              eng.stream())

    for mode in (_lib.SRG_MODE_NOUN, _lib.SRG_MODE_VERB):
        ws = eng.workspace(mode, B, _lib.SRG_PREC_BF16, True)
        for prec, w, g, msg in ((_lib.SRG_PREC_BF16, None, ctypes.byref(sg), b"null workspace"),
                                (_lib.SRG_PREC_BF16, ws, None, b"null argument"),
                                (_lib.SRG_PREC_FP32, ws, ctypes.byref(sg), b"bf16-packed")):
            eng.ensure_packed(m, prec)
            torch.cuda.synchronize()
            before = eng.lib.srg_launch_count()
            assert call(mode, w, g) != 0 and msg in eng.lib.srg_last_error()
            torch.cuda.synchronize()
            assert eng.lib.srg_launch_count() == before
    assert all(t.abs().max() == 0 for t in grads.values()) and dfeat.abs().max() == 0


def test_backbone_gradients_land_in_the_flat_buffer(enc_syn):
    """A trainable ResNet-152 with flat buffers: autograd accumulates its gradients IN PLACE into the `.grad` views of
    the flat buffer (backward runs with grad mode off), so the fused optimizer step sees them."""
    B = 4
    m = S.FCGGNN(enc_syn, 2048, pretrained=False).cuda().train()
    m.convnet_verbs.requires_grad_(True)
    m.convnet_nouns.requires_grad_(True)
    flat = parallel.attach(m, flat_params=True)
    flat.zero()
    img = torch.rand(B, 3, 64, 64, device="cuda")
    gt_verb = torch.randint(0, 504, (B,), device="cuda")
    gt_nouns = torch.randint(0, 2001, (B, 3, 6), device="cuda")
    pv, pn, _ = m(img, gt_verb)
    (m.verb_loss(pv, gt_verb) + m.nouns_loss(pn, gt_nouns)).backward()
    torch.cuda.synchronize()
    lo, hi = flat.flat.data_ptr(), flat.flat.data_ptr() + flat.nbytes()
    ids = {id(p) for p in flat.params}
    for name in ("convnet_verbs", "convnet_nouns"):
        ps = list(getattr(m, name).parameters())
        assert ps and all(id(p) in ids for p in ps)
        for p in ps:
            assert lo <= p.grad.data_ptr() < hi, name
        assert max(p.grad.abs().max().item() for p in ps) > 0, name
    assert len(flat.params) == 20 + 2 * len(list(m.convnet_verbs.parameters()))


def test_launcher_finetune_backbone(tmp_path, capsys, monkeypatch):
    """sr.py --finetune_backbone against a frozen run from the same SRG_SEED on test_launcher's tiny dataset."""
    from situation_recognition_b200 import sr
    from tests.test_launcher import _make_dataset
    _make_dataset(str(tmp_path))
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("SRG_SEED", "7")
    attached = []
    real_attach = parallel.attach
    monkeypatch.setattr(parallel, "attach", lambda *a, **k: attached.append(real_attach(*a, **k)) or attached[-1])
    common = ["--no_pretrained", "--num_workers", "0", "--batch_size", "4"]
    train = common + ["--train_file", "tiny.json", "--epochs", "2"]
    sr.main(train + ["--model_saving_name", "frozen"])
    sr.main(train + ["--model_saving_name", "ft", "--finetune_backbone"])
    out = capsys.readouterr().out
    assert out.count("Model training started!") == 2
    flat = attached[-1]
    for p in flat.params:                              # the last step's gradients, backbones included
        assert flat.flat.data_ptr() <= p.grad.data_ptr() < flat.flat.data_ptr() + flat.nbytes()
    frozen = torch.load(tmp_path / "checkpoints" / "frozen", weights_only=False)
    ft = torch.load(tmp_path / "checkpoints" / "ft", weights_only=False)
    enc = torch.load(tmp_path / "checkpoints" / "encoder", weights_only=False)
    torch.manual_seed(7)             # sr.main builds its model right after seeding
    m0 = S.FCGGNN(enc, 2048, pretrained=False)
    init = m0.state_dict()
    for k in ("convnet_verbs.model.conv1.weight", "convnet_nouns.model.layer4.2.conv3.weight"):
        assert torch.equal(frozen["model_state_dict"][k].cpu(), init[k])
        assert not torch.equal(ft["model_state_dict"][k].cpu(), init[k]), k
    assert not torch.equal(ft["model_state_dict"]["ggsnn.W_p.weight"].cpu(), init["ggsnn.W_p.weight"])
    n_backbone = sum(1 for k, _ in m0.named_parameters() if k.startswith("convnet"))
    osd = ft["optimizer_state_dict"]
    assert len(osd["state"]) == 20 + n_backbone == len(flat.params)
    assert len(frozen["optimizer_state_dict"]["state"]) == 20
    ps = [torch.nn.Parameter(torch.zeros_like(osd["state"][i]["exp_avg"])) for i in range(len(osd["state"]))]
    torch.optim.Adamax(ps, lr=0.002).load_state_dict(osd)
    sr.main(common + ["--resume_model", "ft", "--evaluate_dev"])
    assert "val losses = [v:" in capsys.readouterr().out
    with pytest.raises(SystemExit, match="--finetune_backbone"):
        sr.main(train + ["--epochs", "3", "--resume_model", "ft"])
