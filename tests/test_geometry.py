"""CPU checks of the geometry fixtures (tests/geometry.py) and of srg_create's bounds: D a positive multiple of 256,
R in [1, 8], T in [1, 8], positive vocabulary sizes.  Every refusal happens before the device is touched, so each one
returns its error code and message on a machine without a GPU too."""
import ctypes

import numpy as np
import pytest

from oracle import ggnn_oracle as O
from tests import geometry as GE

# (R, n_verbs, n_roles, n_labels) of tests/test_geometry_gpu.py
VOCABS = [(8, 37, 23, 257), (3, 504, 190, 2001), (6, 129, 40, 511), (1, 11, 5, 13), (5, 300, 90, 4200)]


@pytest.mark.parametrize("R,V,NR,L", VOCABS)
def test_encoder_has_the_requested_geometry(R, V, NR, L):
    train, enc = GE.make_geometry(R, V, NR, L, seed=0)
    assert (enc.get_max_role_count(), enc.get_num_verbs(), enc.get_num_roles(), enc.get_num_labels()) == (R, V, NR, L)
    counts = GE.verb_counts(enc)
    hist = np.bincount(counts, minlength=R + 1)
    assert len(hist) == R + 1 and (hist >= 1).all(), hist          # every count 0..R, 0-role verbs included
    assert sorted(counts.tolist()) == sorted(GE.role_counts(R, V, 0).tolist())
    # the oracle's tables and the device tables agree with the encoder
    t, c = O.build_tables(enc.roles_per_verb, enc.verb_list, enc.role_list)
    v2r, rc = enc.device_tables()
    assert np.array_equal(c, counts) and np.array_equal(rc, counts)
    assert np.array_equal(v2r.reshape(V, R), t) and t.shape == (V, R)
    assert ((t == NR) == (np.arange(R)[None, :] >= counts[:, None])).all()     # pad slots hold the pad role id
    # a 0-role verb's images carry empty frames and only pad targets
    v0 = GE.verbs_with_count(enc, 0)[0]
    img = next(a for a in train.values() if a["verb"] == enc.verb_list[v0])
    assert img["frames"] == [{}, {}, {}]
    assert (enc.get_label_ids(enc.verb_list[v0], img["frames"]) == L).all()
    assert GE.make_geometry(R, V, NR, L, seed=0)[0] == train                    # deterministic


@pytest.mark.parametrize("R,V,NR,L", VOCABS)
def test_crossing_batch(R, V, NR, L):
    """The gt verbs of the crossing batch: every role count, and compact rows that straddle a 256-row tile boundary
    inside one image (at R = 1, where no image owns two rows, a row count past 256)."""
    _, enc = GE.make_geometry(R, V, NR, L, seed=0)
    verbs = GE.crossing_verbs(enc)
    counts = GE.verb_counts(enc)[verbs.numpy()]
    assert set(counts.tolist()) == set(range(R + 1))
    off, rows = GE.compact_rows(counts)
    if R > 1:
        (b,) = GE.straddles(counts)
        assert b == len(verbs) - 1 and off[b] < 256 < off[b] + counts[b]
        assert not GE.straddles(counts[:-1])
    else:
        assert rows == 257 and not GE.straddles(counts)
    fv, fn, gv, gn = GE.make_batch(enc, len(verbs), 256, seed=3, gt_verb=verbs)
    assert fv.shape == fn.shape == (len(verbs), 256) and gn.shape == (len(verbs), 3, R)
    pad = np.arange(R)[None, :] >= counts[:, None]
    assert ((gn.numpy() == L) == pad[:, None, :]).all()


def test_nine_roles_is_a_valid_encoder():
    """The R = 9 fixture the GPU suite feeds to FCGGNN (which must refuse it)."""
    _, enc = GE.make_geometry(9, 12, 12, 20, seed=0)
    assert enc.get_max_role_count() == 9


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from situation_recognition_b200 import _lib
    return _lib.load()


GOOD = dict(D=256, R=6, T=4, V=504, NR=190, L=2001)
REFUSALS = [("D", 0, "D=0"), ("D", 128, "D=128"), ("D", 2050, "D=2050"), ("R", 0, "R=0"), ("R", 9, "R=9"),
            ("T", 0, "T=0"), ("T", 9, "T=9"), ("V", 0, "vocabulary"), ("NR", 0, "vocabulary"), ("L", 0, "vocabulary")]


@pytest.mark.parametrize("field,value,message", REFUSALS)
def test_srg_create_refuses_out_of_bounds(lib, field, value, message):
    args = dict(GOOD, **{field: value})
    h = ctypes.c_void_p()
    rc = lib.srg_create(ctypes.byref(h), 0, args["D"], args["R"], args["T"], args["V"], args["NR"], args["L"])
    err = lib.srg_last_error()
    assert rc != 0 and not h.value, (field, value, rc)
    assert err and message.encode() in err, err
