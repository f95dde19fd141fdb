"""CPU checks of the feature gradients: the two C entry points refuse a null handle before touching a device, and the
launcher's --finetune_backbone flag exists and refuses the forward-only fp32 precision."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from situation_recognition_b200 import _lib
    return _lib.load()


def test_backward_feat_entry_points_reject_null_handle(lib):
    from situation_recognition_b200 import _lib
    g = _lib.SrgGrads()
    ws = ctypes.create_string_buffer(64)
    rc = lib.srg_nouns_backward_feat(None, None, 0, 1, None, None, 2, None, None, None, 0.0, None, 0, ctypes.byref(g),
                                     None, ws, 64, None)
    assert rc != 0 and b"null handle" in lib.srg_last_error()
    rc = lib.srg_verb_backward_feat(None, None, 0, 1, 2, None, 0.0, None, 0, ctypes.byref(g), None, ws, 64, None)
    assert rc != 0 and b"null handle" in lib.srg_last_error()


def test_finetune_backbone_flag():
    from situation_recognition_b200.sr import build_parser
    assert build_parser().parse_args([]).finetune_backbone is False
    assert build_parser().parse_args(["--finetune_backbone"]).finetune_backbone is True


def test_finetune_backbone_refuses_fp32(capsys):
    from situation_recognition_b200 import sr
    with pytest.raises(SystemExit) as e:
        sr.main(["--finetune_backbone", "--precision", "fp32"])
    assert e.value.code == 2                       # argparse's usage error, before anything is loaded
    assert "--finetune_backbone needs --precision bf16" in capsys.readouterr().err
