"""-m gpu: the top-k situation decode (srg_topk_logsoftmax, srg_situation_nouns, FCGGNN.situations_from_features and the
launcher's --topk_situations) on a B200."""
import ctypes
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

import situation_recognition_b200 as S
from oracle import ggnn_oracle as O
from tests.situations_oracle import situations
from situation_recognition_b200 import _lib
from situation_recognition_b200.synthetic import make_batch, make_train_json

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def enc():
    return S.imsitu_encoder(make_train_json(seed=0), verbose=False)


@pytest.fixture(scope="module")
def tables(enc):
    return O.build_tables(enc.roles_per_verb, enc.verb_list, enc.role_list)


def make_model(enc, D, precision, seed=0, compact=True, cta_group=2):
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


# ---------------------------------------------------------------------------------------------- 1. the row kernel
@pytest.mark.parametrize("k", [1, 5, 16])
# n = 5000 spans several 64-value chunks per lane on both load paths (ldl 5120: 16-byte loads; ldl 5003: 4-byte loads),
# so the running sum is rescaled between chunks
@pytest.mark.parametrize("n,ldl", [(504, 512), (2001, 2048), (37, 41), (16, 16), (1000, 1003), (5000, 5120),
                                   (5000, 5003)])
def test_topk_logsoftmax_crafted(n, ldl, k):
    if k > n:
        pytest.skip("k > n")
    g = torch.Generator().manual_seed(n * 100 + k)
    rows = 777
    x = torch.full((rows, ldl), float("nan"))                         # the padding columns must never be read
    core = torch.randint(-6, 6, (rows, n), generator=g).float() / 4   # many exact ties
    core[: rows // 3] = torch.randn(rows // 3, n, generator=g) * 3
    neg = torch.rand(rows, n, generator=g) < 0.3
    neg[:, 0] = False                                                 # every row keeps a finite entry
    core[neg] = -float("inf")
    core[5, 1:] = -float("inf")                                       # a single finite column
    x[:, :n] = core
    # a storage offset of one float: the 16-byte vector path must step aside for a misaligned base
    for base in (x.cuda(), torch.cat([torch.zeros(1), x.reshape(-1)]).cuda()[1:]):
        idx, logp = topk_call(base, ldl, rows, n, k)
        order = torch.sort(core, dim=1, descending=True, stable=True).indices[:, :k]
        assert torch.equal(idx.cpu(), order)
        ref = torch.log_softmax(core.double(), 1).gather(1, order)
        got = logp.cpu().double()
        inf = torch.isinf(ref)
        assert torch.equal(inf, torch.isinf(got)) and (got[inf] < 0).all()
        # 1e-6 absolute; beyond |logp| = 4 fp32 itself cannot hold that (ulp(16) = 1.9e-6): 2^-22 relative there
        err = ((got - ref).abs() / ref.abs().clamp_min(4.0))[~inf].max().item()
        assert err <= 2.0 ** -22, err


def test_topk_logsoftmax_rejects_bad_arguments():
    x = torch.zeros(4, 64, device="cuda")
    for n, k in ((64, 0), (64, 17), (8, 9), (65, 1)):
        with pytest.raises(_lib.SrgError):
            topk_call(x, 64, 4, n, k)


# ---------------------------------------------------------------------------------------------- 2. composition
def check_composition(m, enc, fv, fn, k):
    B, R, L = fn.shape[0], enc.get_max_role_count(), enc.get_num_labels()
    s = m.situations_from_features(fv, fn, k=k)
    assert s.verbs.shape == (B, k) and s.labels.shape == (B, k, R) and s.score.shape == (B, k)
    with torch.no_grad():
        pv = m.predict_verb(fv, B)
        assert torch.equal(s.verbs, torch.sort(pv, dim=1, descending=True, stable=True).indices[:, :k])
        assert (s.verb_logp.double() - torch.log_softmax(pv.double(), 1).gather(1, s.verbs)).abs().max() <= 1e-5
        counts = torch.tensor([enc.get_role_count(v) for v in range(enc.get_num_verbs())], device="cuda")
        real = torch.arange(R, device="cuda")[None, None, :] < counts[s.verbs][:, :, None]
        for j in range(k):
            pn = m.predict_nouns(fn, s.verbs[:, j], B)                                    # [B, R, L]
            am = pn.argmax(-1)
            rj = real[:, j]
            assert torch.equal(s.labels[:, j][rj], am[rj]), j
            lp = torch.log_softmax(pn.double(), -1).gather(-1, am[..., None])[..., 0]
            assert (s.label_logp[:, j][rj].double() - lp[rj]).abs().max() <= 1e-5
    assert (s.labels[~real] == -1).all() and (s.label_logp[~real] == 0).all()
    rescore = s.verb_logp.double() + s.label_logp.double().sum(-1)
    assert (s.score.double() - rescore).abs().max() <= 1e-4
    # k = 1 is column 0 of k = 5, bit for bit (rows of the forward GEMMs are independent, no split-K)
    s1 = m.situations_from_features(fv, fn, k=1)
    for a, b in zip(s1, s):
        assert torch.equal(a, b[:, :1]), "k=1 differs from column 0 of k=%d" % k
    m.check_verbs()


@pytest.mark.parametrize("cta_group", [2, 1])
@pytest.mark.parametrize("compact", [True, False])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_composition_D256(enc, precision, compact, cta_group):
    m, _ = make_model(enc, 256, precision, compact=compact, cta_group=cta_group)
    fv, fn, _, _ = make_batch(enc, 500, 256, seed=11, device="cuda")
    check_composition(m, enc, fv, fn, 5)


@pytest.mark.parametrize("precision,compact,cta_group", [("bf16", True, 2), ("bf16", False, 1), ("fp32", True, 2),
                                                         ("fp32", False, 1)])
def test_composition_D2048_B6144(enc, precision, compact, cta_group):
    m, _ = make_model(enc, 2048, precision, compact=compact, cta_group=cta_group)
    fv, fn, _, _ = make_batch(enc, 6144, 2048, seed=12, device="cuda")
    check_composition(m, enc, fv, fn, 5)


def test_given_verbs_and_argument_checks(enc):
    m, _ = make_model(enc, 256, "bf16")
    fv, fn, gt_verb, _ = make_batch(enc, 64, 256, seed=13, device="cuda")
    s = m.situations_from_features(None, fn, verbs=gt_verb[:, None])
    assert s.verb_logp is None and torch.equal(s.verbs, gt_verb[:, None])
    assert torch.allclose(s.score, s.label_logp.sum(-1))
    with torch.no_grad():
        am = m.predict_nouns(fn, gt_verb, 64).argmax(-1)
    real = s.labels[:, 0] >= 0
    assert torch.equal(s.labels[:, 0][real], am[real])
    m.train()                                          # no dropout and no autograd node in train mode either
    s2 = m.situations_from_features(None, fn, verbs=gt_verb[:, None])
    assert not s2.score.requires_grad and torch.equal(s2.labels, s.labels) and torch.equal(s2.score, s.score)
    m.eval()
    for k in (0, 17, 505):
        with pytest.raises(_lib.SrgError):
            m.situations_from_features(fv, fn, k=k)
    s3 = m.predict_situations(fv, k=3, img_nouns=fn)
    for a, b in zip(s3, m.situations_from_features(fv, fn, k=3)):
        assert torch.equal(a, b)


def test_situation_nouns_workspace_at_any_16_byte_offset(enc):
    """srg_situation_nouns through the C ABI with a workspace of exactly srg_situation_workspace_bytes that does not
    start on a 1024-byte boundary (allocators guarantee 256, 512 or 16 bytes): same results as the aligned call."""
    m, _ = make_model(enc, 256, "bf16")
    fv, fn, _, _ = make_batch(enc, 96, 256, seed=18, device="cuda")
    ref = m.situations_from_features(fv, fn, k=5)
    eng = m._engine_for(fn.device)
    B, k, R = 96, 5, eng.R
    need = eng.lib.srg_situation_workspace_bytes(eng.h, B, k, 0)
    buf = torch.empty(need + 2048, dtype=torch.uint8, device="cuda")
    base = (-buf.data_ptr()) % 1024                                 # first 1024-aligned byte of the buffer
    for extra in (0, 512, 16):
        buf.fill_(0xFF)
        ws = ctypes.c_void_p(buf.data_ptr() + base + extra)
        labels = torch.empty(B, k, R, dtype=torch.int64, device="cuda")
        lp = torch.empty(B, k, R, dtype=torch.float32, device="cuda")
        score = torch.empty(B, k, dtype=torch.float32, device="cuda")
        _lib.check(eng.lib.srg_situation_nouns(eng.h, _lib.ptr(fn), _lib.ptr(ref.verbs), B, k,
                                               _lib.ptr(m.role_emb.weight), _lib.ptr(m.verb_emb.weight),
                                               _lib.ptr(ref.verb_logp), _lib.ptr(labels), _lib.ptr(lp), _lib.ptr(score),
                                               0, ws, need, eng.stream()))
        assert torch.equal(labels, ref.labels) and torch.equal(lp, ref.label_logp) and torch.equal(score, ref.score)
    with pytest.raises(_lib.SrgError):                              # one byte short is refused
        _lib.check(eng.lib.srg_situation_nouns(eng.h, _lib.ptr(fn), _lib.ptr(ref.verbs), B, k,
                                               _lib.ptr(m.role_emb.weight), _lib.ptr(m.verb_emb.weight), None,
                                               _lib.ptr(labels), _lib.ptr(lp), _lib.ptr(score), 0,
                                               ctypes.c_void_p(buf.data_ptr() + base), need - 1, eng.stream()))


# ---------------------------------------------------------------------------------------------- 3. fp32 vs oracle
def test_fp32_parity_vs_oracle(enc, tables):
    B, D, k = 64, 2048, 5
    m, params = make_model(enc, D, "fp32", seed=2)
    fv, fn, _, _ = make_batch(enc, B, D, seed=14)
    s = m.situations_from_features(fv.cuda(), fn.cuda(), k=k)
    t, c = tables
    pv = O.predict_verb(params, fv)
    scale = pv.abs().max().item()
    srt = torch.sort(pv, dim=1, descending=True, stable=True).values[:, :k + 1]
    ok_v = ((srt[:, :-1] - srt[:, 1:]) >= 1e-4 * scale).all(1)
    ov, ovl, _, _, _ = situations(params, fv, fn, k, t, c)
    same_v = (s.verbs.cpu() == ov).all(1)
    assert same_v[ok_v].float().mean().item() >= 0.999
    assert (s.verb_logp.cpu().double() - ovl)[ok_v].abs().max().item() <= 1e-4
    # labels: the oracle conditioned on the CUDA verbs
    cv = s.verbs.cpu()
    _, _, ol, oll, osc = situations(params, fv, fn, k, t, c, verbs=cv)
    ok_l = torch.ones(B, k, dtype=torch.bool)
    for j in range(k):
        nl = O.predict_nouns(params, fn, cv[:, j], t, c)
        top2 = torch.topk(nl, 2, -1).values
        real = torch.arange(nl.shape[1])[None, :] < torch.as_tensor(c)[cv[:, j]][:, None]
        tight = ((top2[..., 0] - top2[..., 1]) < 1e-4 * nl.abs().max().item()) & real
        ok_l[:, j] = ~tight.any(1)
    same_l = (s.labels.cpu() == ol).all(-1)
    frac = same_l[ok_l].float().mean().item()
    print("situations fp32 parity: %d/%d verb rows and %d/%d candidates excluded as near ties; label agreement %.4f"
          % ((~ok_v).sum().item(), B, (~ok_l).sum().item(), B * k, frac))
    assert frac >= 0.999
    assert (s.label_logp.cpu().double() - oll)[ok_l].abs().max().item() <= 1e-4
    rescore = s.verb_logp.cpu().double() + oll.sum(-1)
    assert (s.score.cpu().double() - rescore)[ok_l].abs().max().item() <= 1e-3


# ---------------------------------------------------------------------------------------------- 4. CUDA graph
def test_cuda_graph_replay(enc):
    m, _ = make_model(enc, 256, "bf16")
    B = 512
    fv, fn, _, _ = make_batch(enc, B, 256, seed=15, device="cuda")
    sv, sn = fv.clone(), fn.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        m.situations_from_features(sv, sn, k=5)                  # packs the weights before the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = m.situations_from_features(sv, sn, k=5)
    for seed in (16, 17):
        nv, nn_, _, _ = make_batch(enc, B, 256, seed=seed, device="cuda")
        sv.copy_(nv)
        sn.copy_(nn_)
        g.replay()
        eager = m.situations_from_features(nv, nn_, k=5)
        for a, b in zip(out, eager):
            assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------- 5. launcher
def _lines(out, start):
    """The non-empty output lines from the first one that starts with `start` (the encoder is built, and reports
    itself, on the first run only)."""
    lines = [l for l in out.splitlines() if l.strip()]
    return lines[[i for i, l in enumerate(lines) if l.startswith(start)][0]:]


def test_launcher_topk_situations(tmp_path, capsys, monkeypatch):
    from situation_recognition_b200 import sr
    from tests.test_launcher import _make_dataset
    first = _make_dataset(str(tmp_path))
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("SRG_SEED", "7")
    common = ["--no_pretrained", "--num_workers", "0", "--batch_size", "4"]
    sr.main(common + ["--evaluate_dev"])
    base = _lines(capsys.readouterr().out, "=> evaluating")
    sr.main(common + ["--evaluate_dev", "--topk_situations", "5"])
    out = _lines(capsys.readouterr().out, "=> evaluating")
    assert out[:len(base)] == base                       # the existing lines are unchanged
    block = out[len(base):]
    assert block[0] == "top-k situations (imSitu definitions):"
    assert block[1].startswith("top-1: verb: ") and block[2].startswith("top-5: verb: ")
    assert block[3].startswith("gt-value: ") and "mean = " in block[3]
    img = os.path.join("resized_256", first)
    sr.main(common + ["--test_img", img])
    base = _lines(capsys.readouterr().out, "Using ")
    sr.main(common + ["--test_img", img, "--topk_situations", "3"])
    out = _lines(capsys.readouterr().out, "Using ")
    assert out[:len(base)] == base
    heads = [l for l in out if l.startswith("situation ")]
    assert [h.split()[1] for h in heads] == ["1", "2", "3"] and all("%)" in h for h in heads)
    sr.main(common + ["--test_img", img, "--verb", "verb003", "--topk_situations", "3"])
    heads = [l for l in capsys.readouterr().out.splitlines() if l.startswith("situation ")]
    assert heads == [h for h in heads if "(given): verb003" in h] and len(heads) == 1


_DUMP = """import json, sys
from situation_recognition_b200 import sr
orig = sr._print_situation_scores
def dump(sit):
    orig(sit)
    if sr._rank_world()[0] == 0:
        with open(sys.argv[1], "w") as f:
            json.dump(sit.get_average_results(), f)
sr._print_situation_scores = dump
sr.main(sys.argv[2:])
"""


def _free_port():
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def test_launcher_topk_situations_two_ranks(tmp_path):
    from tests.test_launcher import _make_dataset
    _make_dataset(str(tmp_path))
    script = tmp_path / "dump_eval.py"
    script.write_text(_DUMP)
    args = ["--no_pretrained", "--num_workers", "0", "--batch_size", "4", "--evaluate_dev", "--topk_situations", "5"]
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), SRG_SEED="7")
    if torch.cuda.device_count() < 2:
        env["SRG_DIST_BACKEND"] = "gloo"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), str(script), str(tmp_path / "two.json")] + args
    res = subprocess.run(cmd, cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert res.stdout.count("top-k situations (imSitu definitions):") == 1          # rank 0 prints once
    res1 = subprocess.run([sys.executable, str(script), str(tmp_path / "one.json")] + args, cwd=str(tmp_path), env=env,
                          capture_output=True, text=True, timeout=900)
    assert res1.returncode == 0, res1.stdout[-3000:] + res1.stderr[-3000:]
    two, one = json.loads((tmp_path / "two.json").read_text()), json.loads((tmp_path / "one.json").read_text())
    assert set(two) == set(one) and len(one) == 9
    for key in one:
        assert abs(two[key] - one[key]) <= 1e-12, (key, two[key], one[key])
