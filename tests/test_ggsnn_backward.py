"""CPU checks of the GGSNN.forward backward: the C entry point's argument checks and the Python entry's refusal of
CPU tensors, both of which run before anything touches a device."""
import ctypes

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from situation_recognition_b200 import _lib
    return _lib.load()


def test_ggnn_backward_rejects_null_handle(lib):
    from situation_recognition_b200 import _lib
    g = _lib.SrgGrads()
    ws = ctypes.create_string_buffer(64)
    rc = lib.srg_ggnn_backward(None, _lib.SRG_MODE_NOUN, None, None, None, None, 2, ctypes.byref(g), ws, 64, None)
    assert rc != 0 and b"null handle" in lib.srg_last_error()
    rc = lib.srg_ggnn_backward(None, _lib.SRG_MODE_VERB, None, None, None, None, 0, None, None, 0, None)
    assert rc != 0 and lib.srg_last_error()


@pytest.mark.parametrize("verb", [False, True])
def test_cpu_hidden_state_raises_with_grad(lib, verb):
    import situation_recognition_b200 as S
    from situation_recognition_b200 import _lib
    from situation_recognition_b200.synthetic import make_train_json
    enc = S.imsitu_encoder(make_train_json(seed=0, images_per_verb=1), verbose=False)
    m = S.FCGGNN(enc, 256, backbone=None)
    R = enc.get_max_role_count()
    hidden = torch.zeros(2 if verb else 2 * R, 256, requires_grad=True)
    mask = None if verb else torch.ones(2, R, R, requires_grad=True)
    with pytest.raises(_lib.SrgError, match="no CPU path"):
        m.ggsnn(hidden, mask=mask, verb=verb)
