"""ctypes binding of libemphases_b200.so (the C ABI in include/emphases_b200.h).

There is no CPU fallback: if the shared library is missing or fails to load,
every call raises.  Build it with `python -m emphases_b200.build`.
"""
import contextlib
import ctypes
import threading
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# EMPHASES_B200_LIB selects an alternative build (kernel tuning experiments)
LIB_PATH = os.environ.get(
    'EMPHASES_B200_LIB', os.path.join(HERE, 'libemphases_b200.so'))

# include/emphases_b200.h constants
ACT_NONE, ACT_RELU, ACT_GELU, ACT_LEAKY_RELU, ACT_SILU = 0, 1, 2, 3, 4
POOL = {'average': 0, 'max': 1, 'sum': 2, 'center': 3}
HEAD_LOGITS, HEAD_SIGMOID, HEAD_CLAMP = 0, 1, 2
PREC_FP32, PREC_BF16_TC, PREC_BF16X3_TC, PREC_BF16X6_TC = 0, 1, 2, 3
# dropout site kinds (EMPH_DROPOUT_*)
(DROPOUT_POSITIONAL, DROPOUT_ATTENTION, DROPOUT_RESIDUAL1, DROPOUT_FEEDFORWARD,
 DROPOUT_RESIDUAL2, DROPOUT_CONV) = range(6)


def dropout_site(stack, layer, kind, head=0):
    """EMPH_DROPOUT_SITE: stack 0 = frame encoder, 1 = word decoder"""
    return (stack << 24) | (layer << 16) | (kind << 8) | head

_P = ctypes.c_void_p
_I = ctypes.c_int32
_F = ctypes.c_float
_U32 = ctypes.c_uint32
_U64 = ctypes.c_uint64

# name -> argtypes; every function returns int.  Keep in sync with the header
# (tests/test_abi.py checks that every declared symbol is exported).
SIGNATURES = {
    'emph_row_index': [_P, _P, _I, _P, _I, _P],
    'emph_logmel_f32': [_P, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _I, _I, _P, _P],
    'emph_logmel_i16': [_P, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _I, _I, _P, _P],
    'emph_logmel_resampled_f32': [
        _P, _P, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _I, _I, _P, _P, _P, _I, _I, _I, _P, _P],
    'emph_logmel_resampled_i16': [
        _P, _P, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _I, _I, _P, _P, _P, _I, _I, _I, _P, _P],
    'emph_conv_stack': [_P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _P, _P],
    'emph_conv_stack_pool': [
        _P, _P, _I, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P],
    'emph_pack_conv_weights': [_P, _I, _I, _I, _P, _P],
    'emph_pack_conv_weights_adjoint': [_P, _I, _I, _I, _P, _P],
    'emph_pack_conv_weights_tc': [_P, _P, _I, _I, _I, _I, _P, _P],
    'emph_pool_words': [_P, _I, _P, _P, _P, _P, _P, _I, _I, _P, _P],
    'emph_output_head': [_P, _P, _I, _I, _I, _P, _F, _I, _P, _P, _P],
    'emph_pack_rows': [_P, _I, _I, _I, _P, _P, _P, _I, _P, _P],
    'emph_unpack_rows': [_P, _P, _P, _I, _I, _I, _P, _P],
    'emph_widen_rows': [_P, _I, _I, _I, _P, _P],
    'emph_segment_rows': [_P, _I, _P, _P, _P, _I, _P, _I, _P, _P],
    'emph_add_positional': [_P, _P, _P, _I, _I, _P, _I, _P, _P],
    'emph_attention_rows': [_P, _P, _P, _I, _I, _P, _P, _P, _P, _I, _P, _P, _I, _F, _P, _P],
    'emph_transformer_qkv': [_P, _I, _I, _P, _P, _I, _I, _P, _P, ctypes.c_int64, _P],
    'emph_attention_rows_staged': [
        _P, _P, ctypes.c_int64, _I, _I, _P, _P, _P, _I, _P, _P, _I, _F, _I, _P, _P],
    'emph_transformer_proj_norm': [_P, _P, _I, _I, _P, _P, _I, _P, _P, _F, _P, _P, _P],
    'emph_transformer_ffn_norm': [_P, _I, _I, _P, _P, _I, _P, _P, _F, _P, _P, _P],
    'emph_transformer_layer_tail': [
        _P, _P, _I, _I, _P, _P, _I, _P, _P, _P, _P, _F, _P, _P, _P],
    'emph_attention_rows_tc': [
        _P, _P, _P, _I, _I, _P, _P, _P, _P, _I, _P, _P, _I, _F, _I, _P, ctypes.c_int64, _P, _P],
    'emph_add_layernorm': [_P, _P, _P, _P, _F, _P, _I, _I, _P, _P],
    'emph_resample_f32': [_P, ctypes.c_int64, _P, _I, _I, _I, _P, ctypes.c_int64, _P],
    'emph_resample_packed_i16': [
        _P, _P, _P, _P, _P, _I, _P, _I, _I, _I, _P, ctypes.c_int64, _P],
    'emph_resample_packed_f32': [
        _P, _P, _P, _P, _P, _I, _P, _I, _I, _I, _P, ctypes.c_int64, _P],
    'emph_activation_backward': [_P, _P, _P, _I, _I, _I, _P, _P],
    'emph_activation_forward': [_P, _P, _I, _I, _I, _P, _P],
    'emph_conv_weight_grad': [_P, _P, _I, _I, _I, _P, _P, _P],
    'emph_pool_words_backward': [_P, _P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P],
    'emph_output_head_backward': [_P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P],
    'emph_masked_loss': [_P, _P, _P, _I, _I, _P, _P, _P],
    'emph_upsample_words': [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    'emph_dropout_keep': [_U64, _U32, _U64, ctypes.c_int64, _F, _P, _P],
    'emph_dropout_rows': [_P, _I, _I, _U64, _U32, _F, _P, _P],
    'emph_conv_dropout_forward': [_P, _P, _P, _I, _I, _I, _I, _U64, _U32, _F, _P, _P],
    'emph_activation_dropout_backward': [
        _P, _P, _P, _P, _I, _I, _I, _I, _U64, _U32, _F, _P, _P],
    'emph_linear_rows': [_P, _I, _I, _P, _P, _I, _I, _P, _P, _P],
    'emph_linear_rows_backward': [_P, _I, _I, _P, _I, _P, _P, _P, _P],
    'emph_attention_rows_train': [
        _P, _P, _P, _I, _I, _P, _P, _P, _P, _I, _P, _P, _I, _F, _U64, _U32, _F, _P, _P, _P],
    'emph_attention_rows_backward': [
        _P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _I, _P, _P, _I, _P, _P, _I, _F, _U64, _U32,
        _F, _P, _P, _P, _P],
    'emph_add_layernorm_train': [
        _P, _P, _P, _P, _F, _P, _I, _I, _U64, _U32, _F, _P, _P, _P, _P],
    'emph_layernorm_backward_blocks': [_I],
    'emph_add_layernorm_backward': [
        _P, _P, _P, _P, _P, _I, _I, _U64, _U32, _F, _P, _P, _P, _P, _P, _P],
    'emph_word_metric_sums': [
        _P, _P, _P, _P, _I, _I, _I, ctypes.c_double, ctypes.c_double, _P, _P],
}

class UtteranceStack(ctypes.Structure):
    """emph_utterance_stack"""
    _fields_ = [
        ('weights', _P), ('bias', _P), ('acts_host', _P), ('n_layers', _I),
        ('channels', _I), ('kernel_size', _I), ('precision', _I)]


class UtteranceModel(ctypes.Structure):
    """emph_utterance_model"""
    _fields_ = [
        ('frame', UtteranceStack), ('word', UtteranceStack), ('has_word_stack', _I),
        ('head_weight', _P), ('head_bias', _F), ('head_kernel', _I), ('head_mode', _I),
        ('mel_ptr', _P), ('mel_col', _P), ('mel_val', _P), ('n_mels', _I),
        ('normalize', _I), ('pool_method', _I)]


class TrainModel(ctypes.Structure):
    """emph_train_model"""
    _fields_ = [
        ('n_frame_layers', _I), ('n_word_layers', _I), ('channels', _I),
        ('kernel_size', _I), ('head_kernel', _I), ('pool_method', _I),
        ('forward_precision', _I), ('precision', _I),
        ('acts', _P), ('weights', _P), ('biases', _P), ('zero_bias', _P),
        ('dropout', _P), ('seed', _U64)]


ENOSYS = -38        # EMPH_ENOSYS: the configuration is not built / not handled

_lib = None


class EmphasesB200Error(RuntimeError):
    pass


def load():
    """Load the shared library once; raise loudly when it is absent"""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EmphasesB200Error(
            f'{LIB_PATH} is missing: run `python -m emphases_b200.build`. '
            'emphases_b200 has no CPU or PyTorch fallback path.')
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int
    lib.emph_version.restype = ctypes.c_int
    lib.emph_last_error.restype = ctypes.c_char_p
    lib.emph_device_sm_count.restype = ctypes.c_int
    lib.emph_corpus_fill_files.argtypes = [_P, _P, _I, _P, _P, _P, _P, _I]
    lib.emph_corpus_fill_files.restype = ctypes.c_int
    lib.emph_pack_audio_f32.argtypes = [_P, _P, _P, _I, _P, _P, _P, _I]
    lib.emph_pack_audio_f32.restype = ctypes.c_int
    lib.emph_write_score_rows.argtypes = [_P, _P, _P, _I, _I]
    lib.emph_write_score_rows.restype = ctypes.c_int
    lib.emph_write_score_files.argtypes = [_P, _P, _P, _P, _I, _I]
    lib.emph_write_score_files.restype = ctypes.c_int
    lib.emph_corpus_open.argtypes = [_P, _P, _I, _I]
    lib.emph_corpus_open.restype = ctypes.c_void_p
    lib.emph_corpus_open_blob.argtypes = [ctypes.c_char_p, ctypes.c_char_p, _I, _I]
    lib.emph_corpus_open_blob.restype = ctypes.c_void_p
    lib.emph_corpus_write_textgrids_blob.argtypes = [_P, ctypes.c_char_p, _P, _I]
    lib.emph_corpus_write_textgrids_blob.restype = ctypes.c_int
    lib.emph_write_score_rows_blob.argtypes = [ctypes.c_char_p, _P, _P, _P, _I, _I]
    lib.emph_write_score_rows_blob.restype = ctypes.c_int
    lib.emph_file_sizes.argtypes = [ctypes.c_char_p, _I, _I, _P]
    lib.emph_file_sizes.restype = ctypes.c_int
    lib.emph_corpus_info.argtypes = [_P, _P, _P, _P, _P, _P]
    lib.emph_corpus_info.restype = ctypes.c_int
    lib.emph_corpus_error.argtypes = [_P, _I]
    lib.emph_corpus_error.restype = ctypes.c_char_p
    lib.emph_corpus_fill.argtypes = [_P, _P, _P, _P, _P, _I]
    lib.emph_corpus_fill.restype = ctypes.c_int
    lib.emph_corpus_write_textgrids.argtypes = [_P, _P, _I]
    lib.emph_corpus_write_textgrids.restype = ctypes.c_int
    lib.emph_corpus_close.argtypes = [_P]
    lib.emph_corpus_close.restype = None
    lib.emph_conv_weights_tc_bytes.argtypes = [_I, _I, _I, _I]
    lib.emph_conv_weights_tc_bytes.restype = ctypes.c_int
    lib.emph_attention_tc_workspace.argtypes = [_I, _I, _I, _I]
    lib.emph_attention_tc_workspace.restype = ctypes.c_int64
    lib.emph_infer_utterance_workspace.argtypes = [ctypes.c_longlong, _I, _I, _I]
    lib.emph_infer_utterance_workspace.restype = ctypes.c_longlong
    lib.emph_infer_utterance.argtypes = [
        ctypes.POINTER(UtteranceModel), _P, _I, _P, _I, ctypes.c_longlong, _P,
        ctypes.c_longlong, ctypes.POINTER(_P), ctypes.POINTER(_P), _P]
    lib.emph_infer_utterance.restype = ctypes.c_int
    lib.emph_train_workspace.argtypes = [ctypes.POINTER(TrainModel), _I, _I, _I]
    lib.emph_train_workspace.restype = ctypes.c_longlong
    lib.emph_train_forward.argtypes = [
        ctypes.POINTER(TrainModel), _P, _I, _I, _P, _P, _P, _I, _P, ctypes.c_longlong, _P, _P]
    lib.emph_train_forward.restype = ctypes.c_int
    lib.emph_train_backward.argtypes = [
        ctypes.POINTER(TrainModel), _P, _I, _I, _P, _I, _P, ctypes.c_longlong, _P, _I, _P]
    lib.emph_train_backward.restype = ctypes.c_int
    _lib = lib
    return lib


def call(name, *args):
    """Call an entry point; non-zero status -> EmphasesB200Error"""
    lib = load()
    status = getattr(lib, name)(*args)
    if status != 0:
        message = lib.emph_last_error().decode('utf-8', 'replace')
        raise EmphasesB200Error(f'{name} failed ({status}): {message}')


def ptr(tensor):
    """Device pointer of a torch tensor (None -> NULL)"""
    if tensor is None:
        return None
    return ctypes.c_void_p(tensor.data_ptr())


_pinned_stream = threading.local()


def stream_ptr(stream=None):
    import torch
    if stream is None:
        cached = getattr(_pinned_stream, 'handle', None)
        if cached is not None:
            return cached
        stream = torch.cuda.current_stream()
    return ctypes.c_void_p(stream.cuda_stream)


@contextlib.contextmanager
def same_stream():
    """Within the block every launch of this thread goes to the stream that is
    current on entry: torch.cuda.current_stream() costs ~15 us per lookup,
    more than a small launch (a single-utterance call makes a dozen)."""
    import torch
    previous = getattr(_pinned_stream, 'handle', None)
    _pinned_stream.handle = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    try:
        yield
    finally:
        _pinned_stream.handle = previous
