"""ctypes binding of libsrggnn.so (include/srggnn.h).  There is no fallback: if the shared object is missing
or a call fails, an exception is raised."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SRG_LIB_PATH: load another build of the library (A/B measurements of two revisions on the same GPU box)
LIB_PATH = os.environ.get("SRG_LIB_PATH") or os.path.join(_HERE, "libsrggnn.so")

SRG_DT_F32, SRG_DT_BF16 = 1, 2
SRG_PREC_BF16, SRG_PREC_FP32 = 0, 1
SRG_MODE_NOUN, SRG_MODE_VERB = 0, 1

_c = ctypes
_vp, _i, _i64, _f, _sz = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_float, _c.c_size_t

_PARAM_FIELDS = ["W_p", "b_p", "W_z", "b_Wz", "U_z", "b_Uz", "W_r", "b_Wr", "U_r", "b_Ur", "W_h", "b_Wh", "U_h",
                 "b_Uh", "Wc_verb", "bc_verb", "Wc_noun", "bc_noun"]


class SrgParams(_c.Structure):
    _fields_ = [(n, _vp) for n in _PARAM_FIELDS]


class SrgGrads(_c.Structure):
    _fields_ = [(n, _vp) for n in _PARAM_FIELDS + ["role_emb", "verb_emb"]]


SRG_REDUCTION = {"mean": 0, "sum": 1, "none": 2}


class SrgLossOpts(_c.Structure):
    _fields_ = [("class_weight", _vp), ("label_smoothing", _f), ("reduction", _i), ("per_target_loss", _vp),
                ("grad_per_target", _vp)]


# name -> (restype, argtypes); mirrors include/srggnn.h one to one
SIGNATURES = {
    "srg_last_error": (_c.c_char_p, []),
    "srg_version": (_i, []),
    "srg_create": (_i, [_c.POINTER(_vp), _i, _i, _i, _i, _i, _i, _i]),
    "srg_destroy": (_i, [_vp]),
    "srg_set_cta_group": (_i, [_vp, _i]),
    "srg_set_compact_rows": (_i, [_vp, _i]),
    "srg_set_tables": (_i, [_vp, _vp, _vp]),
    "srg_check_verbs": (_i, [_vp, _vp]),
    "srg_gather_mask": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "srg_pack_weights": (_i, [_vp, _c.POINTER(SrgParams), _i, _vp]),
    "srg_workspace_bytes": (_sz, [_vp, _i, _i, _i, _i]),
    "srg_nouns_forward": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _i64, _vp, _i64, _i, _i, _vp, _sz, _vp]),
    "srg_verb_forward": (_i, [_vp, _vp, _i, _vp, _f, _vp, _i64, _vp, _i64, _i, _i, _vp, _sz, _vp]),
    "srg_topk_logsoftmax": (_i, [_vp, _i64, _i, _i, _i, _vp, _vp, _vp]),
    "srg_situation_workspace_bytes": (_sz, [_vp, _i, _i, _i]),
    "srg_situation_nouns": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _sz, _vp]),
    "srg_situation_nbest_workspace_bytes": (_sz, [_vp, _i, _i, _i, _i]),
    "srg_situation_nbest": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp,
                                 _sz, _vp]),
    "srg_dropout_mask": (_i, [_vp, _i64, _f, _i64, _i, _vp, _vp]),
    "srg_ggnn_forward": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _vp, _sz, _vp]),
    "srg_count_targets": (_i, [_vp, _vp, _i, _vp, _vp]),
    "srg_nouns_loss": (_i, [_vp, _vp, _i64, _vp, _i, _vp, _vp, _vp, _f, _vp, _vp]),
    "srg_verb_loss": (_i, [_vp, _vp, _i64, _vp, _i, _f, _vp, _vp, _vp, _f, _vp, _vp]),
    "srg_nouns_loss_backward": (_i, [_vp, _vp, _i64, _vp, _i, _vp, _vp, _f, _vp, _vp, _i, _vp, _vp]),
    "srg_verb_loss_backward": (_i, [_vp, _vp, _i64, _vp, _i, _f, _vp, _vp, _f, _vp, _vp, _i, _vp, _vp]),
    "srg_count_targets_weighted": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "srg_verb_weight_total": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "srg_nouns_loss_ex": (_i, [_vp, _vp, _i64, _vp, _i, _vp, _vp, _vp, _f, _vp, _c.POINTER(SrgLossOpts), _vp]),
    "srg_verb_loss_ex": (_i, [_vp, _vp, _i64, _vp, _i, _f, _vp, _vp, _vp, _f, _vp, _c.POINTER(SrgLossOpts), _vp]),
    "srg_nouns_loss_backward_ex": (_i, [_vp, _vp, _i64, _vp, _i, _vp, _vp, _f, _vp, _vp, _i, _vp,
                                        _c.POINTER(SrgLossOpts), _vp]),
    "srg_verb_loss_backward_ex": (_i, [_vp, _vp, _i64, _vp, _i, _f, _vp, _vp, _f, _vp, _vp, _i, _vp,
                                       _c.POINTER(SrgLossOpts), _vp]),
    "srg_workspace_stats_offset": (_sz, [_vp, _i, _i, _i, _i, _vp]),
    "srg_workspace_dlogits_offset": (_sz, [_vp, _i, _i, _vp]),
    "srg_nouns_backward": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _i64, _c.POINTER(SrgGrads),
                                _vp, _sz, _vp]),
    "srg_verb_backward": (_i, [_vp, _vp, _i64, _i, _i, _vp, _f, _vp, _i64, _c.POINTER(SrgGrads), _vp, _sz, _vp]),
    "srg_nouns_backward_feat": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _i64,
                                     _c.POINTER(SrgGrads), _vp, _vp, _sz, _vp]),
    "srg_verb_backward_feat": (_i, [_vp, _vp, _i64, _i, _i, _vp, _f, _vp, _i64, _c.POINTER(SrgGrads), _vp, _vp, _sz,
                                    _vp]),
    "srg_ggnn_backward": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _c.POINTER(SrgGrads), _vp, _sz, _vp]),
    "srg_set_deferred_chain": (_i, [_vp, _i, _vp]),
    "srg_chain_finalize": (_i, [_vp, _c.POINTER(SrgGrads), _vp]),
    "srg_clip_adamax": (_i, [_vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _vp, _vp]),
    "srg_sumsq": (_i, [_vp, _i64, _vp, _vp]),
    "srg_adamax_step": (_i, [_vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _vp, _vp, _vp]),
    "srg_launch_count": (_c.c_longlong, []),
    "srg_profile_begin": (_i, []),
    "srg_profile_end": (_i, [_i, _vp, _vp, _vp]),
    "srg_profile_kind_name": (_c.c_char_p, [_i]),
    "srg_gemm_bf16": (_i, [_vp, _i64, _i, _vp, _i64, _i, _vp, _i64, _i, _i, _i, _i, _vp, _f, _i, _i, _i, _vp]),
}

_lib = None


class SrgError(RuntimeError):
    pass


def load():
    """Load libsrggnn.so and declare every prototype.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SrgError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU/PyTorch fallback for the GGNN stage)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing -> loud
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().srg_last_error()
        raise SrgError(f"libsrggnn call failed (code {rc}): {msg.decode() if msg else '?'}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    """The current CUDA stream of `device` (default: the current device) as the void* the C ABI takes."""
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
