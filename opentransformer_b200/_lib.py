"""ctypes binding of libotb200.so (C ABI declared in include/otb200.h).

The product path fails loudly when the CUDA library is missing: there is NO CPU / PyTorch fallback.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_uint8, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('OTB_LIB_PATH') or os.path.join(_HERE, 'libotb200.so')   # OTB_LIB_PATH: A/B runs of two builds (tools/)

_lib = None


class BeamStateC(ctypes.Structure):
    """otb_beam_state (include/otb200.h)."""
    _fields_ = [('tok_hist', c_void_p), ('par_hist', c_void_p), ('last_tok', c_void_p), ('scores', c_void_p),
                ('flag', c_void_p), ('anc', c_void_p), ('ctrl', c_void_p),
                ('N', c_int32), ('beam', c_int32), ('Lmax', c_int32)]


class MegaLayerC(ctypes.Structure):
    """otb_mega_layer (include/otb200.h)."""
    _fields_ = [(n, c_void_p) for n in ('wqkv', 'wo', 'wq', 'wo2', 'w1', 'w2', 'bqkv', 'bo', 'bq', 'bo2', 'b1', 'b2',
                                        'g1', 'be1', 'g2', 'be2', 'g3', 'be3')]


MEGA_MAX_LAYERS = 8


class MegaModelC(ctypes.Structure):
    """otb_mega_model (include/otb200.h)."""
    _fields_ = [('n_layers', c_int32), ('d_model', c_int32), ('n_heads', c_int32), ('d_ff', c_int32), ('vocab', c_int32),
                ('emb', c_void_p), ('wout', c_void_p), ('bout', c_void_p), ('pe', c_void_p),
                ('layers', MegaLayerC * MEGA_MAX_LAYERS), ('ln_eps', c_float)]


_P = c_void_p
_SIGS = {
    'otb_last_error': (c_char_p, []),
    'otb_version': (c_int, []),
    'otb_num_sms': (c_int, []),
    'otb_debug_gemm_timing': (c_int, [_P]),
    'otb_debug_gemm_mode': (c_int, [c_int]),
    'otb_set_tile_policy': (c_int, [c_int]),
    'otb_debug_decode_timing': (c_int, [_P, c_int]),
    'otb_set_decode_barrier': (c_int, [c_int]),
    'otb_conv_geometry': (c_int, [c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    'otb_conv1_relu': (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    'otb_conv2_relu': (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    'otb_linear': (c_int, [_P, c_int, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, _P, _P,
                           c_float, c_float, _P, c_int, _P, c_int, _P]),
    'otb_linear_dropout_resid': (c_int, [_P, c_int, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, _P, c_int, c_float, c_float, _P,
                                         ctypes.c_uint32, _P]),
    'otb_dropout_bwd': (c_int, [_P, c_int, _P, c_int, _P, c_int, c_int, c_float, _P, ctypes.c_uint32, _P]),
    'otb_attention': (c_int, [_P, c_int, c_int, _P, c_int, c_int, _P, c_int, _P, c_int, c_int, c_int, c_int, c_int,
                              _P, c_int, c_int, c_int, c_int, _P, c_int, _P, c_int, _P]),
    'otb_dwconv_swish': (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    'otb_layernorm': (c_int, [_P, c_int, _P, c_int, c_int, _P, _P, _P, _P, c_float, c_int, c_int, _P]),
    'otb_scale_add_table': (c_int, [_P, c_int, c_int, _P, c_int, c_float, _P, c_int, c_int, c_int, _P]),
    'otb_sinusoid_table': (c_int, [_P, c_int, c_int, c_int, _P]),
    'otb_embed_posenc': (c_int, [_P, c_int, _P, _P, _P, c_int, c_int, c_int, _P, c_int, _P]),
    'otb_log_softmax': (c_int, [_P, c_int, _P, c_int, c_int, c_int, _P]),
    'otb_decode_self_attn': (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, _P]),
    'otb_decode_self_attn_hd': (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    'otb_ls_ce': (c_int, [_P, c_int, _P, c_int, c_int, c_float, c_int, _P, _P, _P, _P, c_int, _P]),
    'otb_beam_init': (c_int, [POINTER(BeamStateC), _P]),
    'otb_beam_step': (c_int, [_P, c_int, c_int, _P, c_int, c_float, POINTER(BeamStateC), _P, _P, _P]),
    'otb_beam_step_topk': (c_int, [_P, _P, POINTER(BeamStateC), _P, _P, _P]),
    'otb_logsoftmax_topk': (c_int, [_P, c_int, c_int, _P, c_int, c_float, c_int, c_int, _P, _P, _P, c_int, _P]),
    'otb_beam_reconstruct': (c_int, [POINTER(BeamStateC), _P, c_int, c_int, _P]),
    'otb_beam_finalize': (c_int, [POINTER(BeamStateC), c_float, c_float, c_int, _P, _P, _P]),
    'otb_attention_lse': (c_int, [_P, c_int, c_int, _P, c_int, c_int, _P, c_int, _P, c_int, c_int, c_int, c_int, c_int,
                                  _P, c_int, c_int, c_int, c_int, _P, c_int, _P, c_int, _P, _P]),
    'otb_attention_hd': (c_int, [_P, c_int, c_int, _P, c_int, c_int, _P, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                                 _P, c_int, c_int, c_int, c_int, _P, c_int, _P, c_int, _P]),
    'otb_attention_lse_hd': (c_int, [_P, c_int, c_int, _P, c_int, c_int, _P, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                                     _P, c_int, c_int, c_int, c_int, _P, c_int, _P, c_int, _P, _P]),
    'otb_attention_bwd': (c_int, [_P, c_int, c_int, _P, c_int, c_int, _P, c_int, _P, c_int, _P, c_int, _P, _P, _P, c_int, c_int,
                                  _P, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, _P]),
    'otb_linear_wgrad': (c_int, [_P, c_int, _P, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    'otb_colsum': (c_int, [_P, c_int, _P, c_int, c_int, c_int, _P]),
    'otb_layernorm_bwd': (c_int, [_P, c_int, _P, c_int, _P, _P, c_int, _P, _P, c_float, c_int, c_int, c_int, _P]),
    'otb_glu_fwd': (c_int, [_P, _P, c_int, c_int, _P]),
    'otb_glu_bwd': (c_int, [_P, _P, _P, c_int, c_int, _P]),
    'otb_relu_bwd': (c_int, [_P, _P, _P, c_int64, _P]),
    'otb_embed_bwd': (c_int, [_P, _P, _P, c_int, c_int, c_int, c_float, _P]),
    'otb_ls_ce_train': (c_int, [_P, c_int, _P, c_int, c_int, c_float, c_int, _P, _P, _P, _P, c_int, _P]),
    'otb_sumsq': (c_int, [_P, c_int64, _P, c_int, _P]),
    'otb_adam_step': (c_int, [_P, _P, _P, _P, c_int64, _P, c_float, c_float, c_float, c_float, c_float, c_float, c_int, _P]),
    'otb_adam_step_sched': (c_int, [_P, _P, _P, _P, c_int64, _P, c_float, c_float, c_float, c_float, c_float, c_float, c_float,
                                    c_float, c_float, _P, _P, _P]),
    'otb_fbank': (c_int, [_P, c_int, _P, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, _P]),
    'otb_utt_cmvn': (c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P]),
    'otb_ctc_loss': (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, c_int, c_int, _P, _P, _P, _P, c_int, c_float, _P]),
    'otb_conv_im2col': (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    'otb_conv_col2im_relu': (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    'otb_conv1_wgrad': (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    'otb_spec_augment': (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    'otb_decode_persistent_workspace': (c_int64, [c_int, c_int, c_int, c_int, c_int, c_int]),
    'otb_decode_persistent': (c_int, [POINTER(MegaModelC), _P, _P, _P, _P, POINTER(BeamStateC), c_int, c_int, c_int, _P, c_int64,
                                      _P, _P, _P]),
}


def exported_symbols():
    """Names every build of the library must export (checked by tests/test_capi_symbols.py)."""
    return sorted(_SIGS)


def lib():
    """Load (once) and return the ctypes handle; raises if the extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} is missing: build it with `python -m opentransformer_b200.build` '
                '(there is no CPU fallback for the B200 hot path)')
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status, what=''):
    if status != 0:
        msg = lib().otb_last_error().decode('utf-8', 'replace')
        raise RuntimeError(f'libotb200 {what} failed: {msg}')
