"""CPU checks of the loss options (class weights, label smoothing, reductions): the C ABI refuses bad options and null
handles, FCGGNN.verb_loss / nouns_loss validate their keywords before any engine call, sr.py exposes and checks
--label_smoothing / --class_weights, and tools/make_class_weights.py counts through the encoder's ids."""
import ctypes
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from situation_recognition_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def enc():
    import situation_recognition_b200 as S
    from situation_recognition_b200.synthetic import make_train_json
    return S.imsitu_encoder(make_train_json(seed=0, images_per_verb=1), verbose=False)


def _opts(eps=0.0, reduction=0, per_target=None, gpt=None):
    from situation_recognition_b200 import _lib
    return _lib.SrgLossOpts(None, eps, reduction, per_target, gpt)


def _calls(lib, o):
    """The four option-taking loss calls with a NULL handle and dummy (never dereferenced) device pointers."""
    p = ctypes.c_void_p(16)
    yield lib.srg_nouns_loss_ex(None, p, 2048, p, 1, p, p, None, 1.0, None, ctypes.byref(o), None)
    yield lib.srg_verb_loss_ex(None, p, 512, p, 1, 1.0, None, p, None, 1.0, None, ctypes.byref(o), None)
    yield lib.srg_nouns_loss_backward_ex(None, p, 2048, p, 1, p, p, 1.0, p, None, 0, None, ctypes.byref(o), None)
    yield lib.srg_verb_loss_backward_ex(None, p, 512, p, 1, 1.0, None, p, 1.0, p, None, 0, None, ctypes.byref(o), None)


@pytest.mark.parametrize("bad,needle", [(dict(eps=-0.1), b"label_smoothing"), (dict(eps=1.5), b"label_smoothing"),
                                        (dict(eps=float("nan")), b"label_smoothing"),
                                        (dict(reduction=3), b"unknown reduction"),
                                        (dict(reduction=2), b"reduction 'none' needs")])
def test_cabi_refuses_bad_options(lib, bad, needle):
    for rc in _calls(lib, _opts(**bad)):
        assert rc != 0
        assert needle in lib.srg_last_error()


def test_cabi_refuses_null_handles(lib):
    for rc in _calls(lib, _opts(eps=0.1)):
        assert rc != 0 and b"null handle" in lib.srg_last_error()
    p = ctypes.c_void_p(16)
    assert lib.srg_count_targets_weighted(None, p, 1, p, p, None) != 0
    assert b"null handle" in lib.srg_last_error()
    assert lib.srg_verb_weight_total(None, p, 1, p, p, None) != 0
    assert b"null handle" in lib.srg_last_error()


def _model(enc):
    import situation_recognition_b200 as S
    return S.FCGGNN(enc, 256, backbone=None)


@pytest.mark.parametrize("which", ["verb", "nouns"])
def test_python_validates_options_before_the_engine(enc, which):
    from situation_recognition_b200 import _lib
    m = _model(enc)
    V, L, R = enc.get_num_verbs(), enc.get_num_labels(), enc.get_max_role_count()
    if which == "verb":
        logits, gt, n, call = torch.zeros(4, V), torch.zeros(4, dtype=torch.long), V, m.verb_loss
    else:
        logits, gt, n, call = torch.zeros(4, R, L), torch.zeros(4, 3, R, dtype=torch.long), L, m.nouns_loss
    with pytest.raises(_lib.SrgError, match="shape"):
        call(logits, gt, weight=torch.ones(n + 1))
    with pytest.raises(_lib.SrgError, match="shape"):
        call(logits, gt, weight=torch.ones(1, n))
    with pytest.raises(_lib.SrgError, match="float32"):
        call(logits, gt, weight=torch.ones(n, dtype=torch.float64))
    with pytest.raises(_lib.SrgError, match="is on"):
        call(logits, gt, weight=torch.ones(n, device="meta"))
    with pytest.raises(_lib.SrgError, match="require grad"):
        call(logits, gt, weight=torch.ones(n, requires_grad=True))
    with pytest.raises(ValueError, match="reduction"):
        call(logits, gt, reduction="avg")
    for eps in (-0.01, 1.01, float("nan")):
        with pytest.raises(ValueError, match="label_smoothing"):
            call(logits, gt, label_smoothing=eps)


def test_sr_help_lists_the_flags():
    from situation_recognition_b200 import sr
    text = sr.build_parser().format_help()
    assert "--label_smoothing" in text and "--class_weights" in text
    assert "dev losses" in text
    res = subprocess.run([sys.executable, "-m", "situation_recognition_b200.sr", "--help"], cwd=ROOT,
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 0 and "--label_smoothing" in res.stdout and "--class_weights" in res.stdout


def test_class_weights_file_must_match_the_encoder(enc, tmp_path):
    from situation_recognition_b200.sr import load_class_weights
    V, L = enc.get_num_verbs(), enc.get_num_labels()
    good = tmp_path / "good.pt"
    torch.save({"verb": torch.ones(V), "nouns": torch.full((L,), 2.0)}, good)
    v, n = load_class_weights(str(good), enc)
    assert v.shape == (V,) and n.shape == (L,) and float(n[0]) == 2.0
    only = tmp_path / "only.pt"
    torch.save({"nouns": torch.ones(L)}, only)
    assert load_class_weights(str(only), enc)[0] is None
    for i, bad in enumerate([{"verb": torch.ones(V + 1)}, {"nouns": torch.ones(L - 1)}, {"nouns": torch.ones(2, L)},
                             {"labels": torch.ones(L)}, {"verb": -torch.ones(V)}]):
        path = tmp_path / ("bad%d.pt" % i)
        torch.save(bad, path)
        with pytest.raises(ValueError):
            load_class_weights(str(path), enc)


def test_make_class_weights_counts_through_the_encoder(tmp_path):
    import situation_recognition_b200 as S
    from situation_recognition_b200.synthetic import make_train_json
    full = make_train_json(seed=3, images_per_verb=3)
    # counted on a subset: verbs with 0 to 3 images, so the frequencies differ and some classes are never seen
    names = sorted(full)
    train = {k: full[k] for i, k in enumerate(names)
             if i % 4 != 0 and i % 7 != 0 and not full[k]["verb"].endswith("5")}
    paths = tmp_path / "train.json", tmp_path / "encoder.json"
    paths[0].write_text(json.dumps(train))
    paths[1].write_text(json.dumps(full))
    out = tmp_path / "w.pt"
    power = 0.5
    res = subprocess.run([sys.executable, "tools/make_class_weights.py", "--train_json", str(paths[0]),
                          "--encoder_json", str(paths[1]), "--out", str(out), "--power", str(power)], cwd=ROOT,
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    w = torch.load(out)
    enc = S.imsitu_encoder(full, verbose=False)
    V, L = enc.get_num_verbs(), enc.get_num_labels()
    assert w["verb"].shape == (V,) and w["nouns"].shape == (L,) and w["nouns"].dtype == torch.float32
    # the counts, independently: by the encoder's ids of every image's verb and every (annotation, role) label
    vc, lc = torch.zeros(V), torch.zeros(L)
    for item in train.values():
        vc[enc._verb_ids[item["verb"]]] += 1
        for frame in item["frames"]:
            for role in enc.roles_per_verb[item["verb"]]:
                lc[enc.label_list.index(frame[role])] += 1
    for counts, got in ((vc, w["verb"]), (lc, w["nouns"])):
        seen = counts > 0
        assert seen.any() and len(set(counts[seen].tolist())) > 1            # the frequencies differ
        expect = counts[seen].double() ** -power
        expect = expect / expect.mean()
        assert torch.allclose(got[seen].double(), expect, rtol=1e-6)
        assert abs(got[seen].double().mean().item() - 1.0) < 1e-6
        assert torch.all(got[~seen] == 1.0)
    assert (vc == 0).any()                      # verbs of the encoder the subset never shows
    # the file is one sr.py accepts for this encoder
    from situation_recognition_b200.sr import load_class_weights
    load_class_weights(str(out), enc)
