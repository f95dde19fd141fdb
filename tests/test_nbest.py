"""CPU checks of the n-best situation decode: the oracle (tests/nbest_oracle.py) on tiny vocabularies -- the top n
labels of each slot are all an n-best list needs, the best-first search equals enumeration, and a certified beam list
equals the list over all verbs -- plus the C entry point's refusal of a null handle and the launcher's argument
checks."""
import ctypes

import numpy as np
import pytest
import torch

from tests.nbest_oracle import certified, nbest_best_first, nbest_enumerate, rank_lists


def random_image(g, V, R, L, integer):
    """Verb log-probs [V] and per-verb label log-probs [V, R, L], fp32, plus role counts [V] in [0, R].  integer:
    integer-valued log-probs (not normalised), so that many situations tie exactly."""
    if integer:
        vlp = -torch.randint(0, 3, (V,), generator=g).float()
        lp = -torch.randint(0, 3, (V, R, L), generator=g).float()
    else:
        vlp = torch.log_softmax(torch.randn(V, generator=g) * 2, 0)
        lp = torch.log_softmax(torch.randn(V, R, L, generator=g) * 2, -1)
    counts = torch.randint(0, R + 1, (V,), generator=g)
    counts[0] = max(int(counts[0]), 1)
    return vlp, lp, counts


def candidates(vlp, lp, counts, verbs, m=None, given=False):
    """The oracle's candidates for these verbs: each real slot's labels in rank order, the top m of them."""
    out = []
    for v in verbs:
        _, slot_lp = rank_lists(lp[v, :int(counts[v])], m)
        out.append((None if given else np.float32(vlp[v]), slot_lp.numpy()))
    return out


def verb_order(vlp):
    return torch.sort(vlp, descending=True, stable=True).indices.tolist()


@pytest.mark.parametrize("integer", [False, True])
@pytest.mark.parametrize("n", [1, 2, 5, 9])
def test_top_n_labels_suffice_and_best_first_equals_enumeration(n, integer):
    g = torch.Generator().manual_seed(n * 10 + integer)
    for trial in range(12):
        V, R, L = 4, 3, 5
        vlp, lp, counts = random_image(g, V, R, L, integer)
        verbs = verb_order(vlp)[:3]
        for given in (False, True):
            full = nbest_enumerate(candidates(vlp, lp, counts, verbs, given=given), n)
            top = nbest_enumerate(candidates(vlp, lp, counts, verbs, m=min(n, L), given=given), n)
            fast = nbest_best_first(candidates(vlp, lp, counts, verbs, m=min(n, L), given=given), n)
            assert len(full) == n
            # no near-tie exclusion: equal scores, candidates and ranks, entry for entry
            assert top == full, (trial, given)
            assert fast == full, (trial, given)
            assert all(full[i][0] >= full[i + 1][0] for i in range(n - 1))


def test_ties_break_by_candidate_then_ranks():
    lp = np.zeros((2, 3), dtype=np.float32)                 # every assignment scores 0
    got = nbest_enumerate([(np.float32(0), lp), (np.float32(0), lp)], 11)
    assert [(j, ranks) for _, j, ranks in got] == [(0, (a, b)) for a in range(3) for b in range(3)] + [(1, (0, 0)),
                                                                                                     (1, (0, 1))]


def test_scores_are_fp32_sums_in_slot_order():
    lp = np.array([[np.float32(1e-8)], [np.float32(-1.0)]], dtype=np.float32)
    (s, _, _), = nbest_enumerate([(np.float32(1.0), lp)], 1)
    assert s.dtype == np.float32 and s == np.float32(np.float32(1.0 + np.float32(1e-8)) - 1.0) == 0.0


@pytest.mark.parametrize("integer", [False, True])
def test_certified_beam_list_equals_list_over_all_verbs(integer):
    g = torch.Generator().manual_seed(7 + integer)
    V, R, L = 6, 3, 4
    seen = {True: 0, False: 0}
    for trial in range(60):
        vlp, lp, counts = random_image(g, V, R, L, integer)
        order = verb_order(vlp)
        for kv in (1, 2, 4):
            for n in (1, 3, 6):
                everything = nbest_enumerate(candidates(vlp, lp, counts, order, m=n), n)
                beam = nbest_enumerate(candidates(vlp, lp, counts, order[:kv], m=n), n)
                exact = certified(beam, n, vlp[order[kv]])
                seen[exact] += 1
                if exact:
                    assert beam == everything, (trial, kv, n)
    assert seen[True] > 0 and seen[False] > 0, seen


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from situation_recognition_b200 import _lib
    return _lib.load()


def test_nbest_entry_points_reject_null_handle(lib):
    ws = ctypes.create_string_buffer(64)
    rc = lib.srg_situation_nbest(None, None, None, 1, 1, None, None, None, None, 1, None, None, None, None, None, None,
                                 0, ws, 64, None)
    assert rc != 0 and b"null handle" in lib.srg_last_error()
    assert lib.srg_situation_nbest_workspace_bytes(None, 1, 1, 1, 0) == 0


@pytest.mark.parametrize("argv", [["--nbest_situations", "4"],
                                  ["--test_img", "x.jpg", "--nbest_situations", "0"],
                                  ["--test_img", "x.jpg", "--nbest_situations", "17"],
                                  ["--evaluate_dev", "--nbest_situations", "3"]])
def test_launcher_rejects_nbest_situations(argv, capsys):
    """--nbest_situations prints one image's list: it needs --test_img and 1 <= N <= 16.  Refused while parsing,
    before anything touches a GPU."""
    from situation_recognition_b200 import sr
    with pytest.raises(SystemExit) as e:
        sr.main(argv)
    assert e.value.code == 2
    assert "--nbest_situations" in capsys.readouterr().err


def test_launcher_nbest_situations_flag():
    from situation_recognition_b200.sr import build_parser
    assert build_parser().parse_args([]).nbest_situations is None
    assert build_parser().parse_args(["--test_img", "x.jpg", "--nbest_situations", "16"]).nbest_situations == 16
