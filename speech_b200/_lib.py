"""ctypes binding of libspeech_b200.so (the C ABI declared in include/speech_b200.h).

There is NO fallback: if the shared library is missing, or a call returns a non-zero status, a
RuntimeError is raised.  The product path never routes through oracle/ or a CPU implementation.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libspeech_b200.so")

_c_int = ctypes.c_int
_c_ll = ctypes.c_longlong
_c_sz = ctypes.c_size_t
_vp = ctypes.c_void_p
_fl = ctypes.c_float

# name -> (restype, argtypes): every symbol include/speech_b200.h declares
SIGNATURES = {
    "sb_version": (_c_int, []),
    "sb_status_string": (ctypes.c_char_p, [_c_int]),
    "sb_device_info": (_c_int, [_vp, _vp, _vp, _vp]),
    "sb_ctc_workspace_size": (_c_int, [_c_int, _c_int, _c_int, _c_int, ctypes.POINTER(_c_sz)]),
    "sb_ctc_fwd_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int,
                                _c_int, _vp, _vp, _c_sz, _vp]),
    "sb_gemm_bf16_tn": (_c_int, [_vp, _c_ll, _vp, _c_ll, _vp, _c_ll, _vp, _c_int, _c_int, _c_int,
                                 _c_int, _c_int, _c_int, _c_int, _c_int, _vp]),
    "sb_ctc_prefix_beam_workspace_size": (_c_int, [_c_int, _c_int, _c_int, ctypes.POINTER(_c_sz)]),
    "sb_ctc_prefix_beam": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp,
                                    _vp, _c_sz, _vp]),
    "sb_conv_im2col": (_c_int, [_vp, _vp, _fl, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                _c_int, _c_int, _c_int, _vp]),
    "sb_conv_relu_to_bct": (_c_int, [_vp, _vp, _fl, _vp, _c_int, _c_int, _c_int, _c_int, _vp]),
    "sb_conv_dtop": (_c_int, [_vp, _vp, _vp, _fl, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp]),
    "sb_conv_col2im_relu": (_c_int, [_vp, _c_ll, _vp, _vp, _fl, _vp, _vp, _c_int, _c_int, _c_int,
                                     _c_int, _c_int, _c_int, _c_int, _vp]),
    "sb_sumsq_workspace_size": (_c_int, [ctypes.POINTER(_c_sz)]),
    "sb_sumsq": (_c_int, [_vp, _c_ll, _vp, _vp, _vp]),
    "sb_sgd_clip_step": (_c_int, [_vp, _vp, _vp, _vp, _c_ll, _vp, _fl, _fl, _fl, _vp]),
    "sb_s2s_workspace_size": (_c_int, [_c_int, _c_int, _c_int, ctypes.POINTER(_c_sz)]),
    "sb_attn_step": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _fl, _c_int, _c_int, _c_int, _c_int,
                              _c_int, _vp, _vp, _vp, _c_sz, _vp]),
    "sb_s2s_cell_fwd": (_c_int, [_vp, _vp, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                 _c_int, _c_int, _vp]),
    "sb_s2s_attn_fwd": (_c_int, [_vp, _c_int, _vp, _vp, _vp, _vp, _vp, _fl, _c_int, _c_int, _c_int,
                                 _c_int, _c_int, _vp, _vp, _vp, _vp, _c_int, _vp, _c_ll, _vp, _vp,
                                 _vp, _c_int, _c_int, _vp, _c_int, _vp, _vp, _c_sz, _vp]),
    "sb_s2s_dout": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_ll, _c_int, _c_int, _vp]),
    "sb_s2s_attn_bwd": (_c_int, [_vp] * 22 + [_c_int] * 5 + [_vp, _c_sz, _vp]),
    "sb_s2s_cell_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _vp]),
    "sb_s2s_check_done": (_c_int, [_vp, _c_int, _vp, _vp, _c_int, _vp]),
    "sb_s2s_beam_state_size": (_c_int, [ctypes.POINTER(_c_sz)]),
    "sb_s2s_beam_init": (_c_int, [_vp, _vp, _vp, _c_int, _vp]),
    "sb_s2s_beam_select": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _c_int,
                                    _c_int, _c_int, _c_int, _c_int, _vp]),
    "sb_s2s_beam_gather": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _c_int,
                                    _vp]),
    "sb_beam_topk": (_c_int, [_vp, _c_int, _c_int, _vp, _vp, _vp]),
    "sb_rnnt_workspace_size": (_c_int, [_c_int, _c_int, _c_int, ctypes.POINTER(_c_sz)]),
    "sb_rnnt_fwd_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int,
                                 _vp, _vp, _c_sz, _vp]),
    "sb_rnnt_fwd_bwd_compact": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int,
                                         _vp, _vp, _c_sz, _vp]),
    "sb_rnnt_joint_fwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int,
                                   _c_int, _c_int, _vp]),
    "sb_rnnt_joint_dlogits": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int,
                                       _c_int, _c_int, _c_int, _c_int, _vp]),
    "sb_rnnt_joint_build_slab": (_c_int, [_vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int,
                                          _c_int, _vp]),
    "sb_rnnt_joint_reduce_slab": (_c_int, [_vp, _vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int,
                                           _c_int, _c_int, _vp]),
    "sb_rnnt_decode_static_workspace_size": (_c_int, [_c_int, _c_int, _c_int, _c_int,
                                                      ctypes.POINTER(_c_sz)]),
    "sb_rnnt_decode_static": (_c_int, [_vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                       _vp, _vp, _vp, _vp, _c_sz, _vp]),
    "sb_debug_gru_timeline": (_c_int, [_vp]),
    "sb_debug_gru_cluster": (_c_int, [_c_int]),
    "sb_edit_distance": (_c_ll, [_vp, _c_ll, _vp, _c_ll]),
    "sb_log_specgram": (_c_int, [_vp, _vp, _vp, _c_int, _c_int, _c_int, ctypes.c_double, _fl, _vp,
                                 _vp, _vp, _c_int, _vp]),
    "sb_gru_fwd_workspace_size": (_c_int, [_c_int, _c_int, _c_int, ctypes.POINTER(_c_sz)]),
    "sb_gru_fwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_sz, _c_int, _c_int, _c_int,
                            _c_int, _vp]),
    "sb_gru_fwd_f32": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp]),
    "sb_gru_bwd_workspace_size": (_c_int, [_c_int, _c_int, _c_int, ctypes.POINTER(_c_sz)]),
    "sb_gru_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_sz, _c_int, _c_int,
                            _c_int, _c_int, _vp]),
}

_lib = None
launch_count = 0   # C-ABI kernel launches issued by this process (bench.py: gpu_launches)


class SpeechB200Error(RuntimeError):
    pass


def load():
    """Load the CUDA library; raises if it has not been built (python -m speech_b200.csrc.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SpeechB200Error(
            "speech_b200: %s is missing - build it with `python -m speech_b200.csrc.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what):
    if status != 0:
        msg = load().sb_status_string(status).decode()
        raise SpeechB200Error("speech_b200: %s failed: %s (status %d)" % (what, msg, status))


def ptr(t):
    """Raw device/host pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t, name):
    if not t.is_cuda:
        raise SpeechB200Error(
            "speech_b200: %s must live on a CUDA device - this package has no CPU path" % name)
