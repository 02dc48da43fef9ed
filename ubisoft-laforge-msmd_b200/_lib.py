"""ctypes binding of libmsmd_b200.so (include/msmd_b200.h).

The library is the product: if it is missing or a symbol is absent we raise —
there is no CPU / eager-PyTorch fallback anywhere in this package.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libmsmd_b200.so')

_vp, _i, _i64 = C.c_void_p, C.c_int, C.c_int64

# name -> (restype, argtypes); mirrors include/msmd_b200.h one to one.
SIGNATURES = {
    'msmd_last_error': (C.c_char_p, []),
    'msmd_version': (C.c_char_p, []),
    'msmd_profile_enable': (_i, [_i]),
    'msmd_profile_reset': (_i, []),
    'msmd_profile_query': (_i, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(_i64)]),
    'msmd_profile_dump': (_i, [C.c_char_p, _i64]),
    'msmd_rot_convert': (_i, [_i, _vp, _vp, _i64, _i, _vp]),
    'msmd_quat_binary': (_i, [_i, _vp, _vp, _vp, _i64, _vp]),
    'msmd_linear': (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i64, _i64, _i64, _i64, _i, _i, _i, _vp]),
    'msmd_split_tf32': (_i, [_vp, _vp, _vp, _i64, _vp]),
    'msmd_split_f16': (_i, [_vp, _vp, _vp, _i64, _vp]),
    'msmd_create': (_i, [_vp, _i, C.POINTER(_vp)]),
    'msmd_destroy': (None, [_vp]),
    'msmd_load_weights': (_i, [_vp, C.POINTER(C.c_char_p), C.POINTER(_vp), C.POINTER(_i64), _i]),
    'msmd_window_begin': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'msmd_denoise': (_i, [_vp, _vp, _vp, _vp, _vp]),
    'msmd_denoise_ex': (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    'msmd_denoise_parts': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    'msmd_check': (_i, [_vp, _vp]),
    'msmd_sample_window': (_i, [_vp, _vp, _vp, C.c_uint64, _i, C.c_float, C.c_float, C.c_float, _i, _i, _vp, _vp, _vp]),
    'msmd_style_create': (_i, [_i, _i, _i, _i, _i, _i, C.POINTER(_vp)]),
    'msmd_style_destroy': (None, [_vp]),
    'msmd_style_load_weights': (_i, [_vp, C.POINTER(C.c_char_p), C.POINTER(_vp), C.POINTER(_i64), _i]),
    'msmd_style_encode': (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    'msmd_audio_create': (_i, [_i, _i, _i, _i, C.POINTER(_vp)]),
    'msmd_audio_destroy': (None, [_vp]),
    'msmd_audio_load_weights': (_i, [_vp, C.POINTER(C.c_char_p), C.POINTER(_vp), C.POINTER(_i64), _i]),
    'msmd_audio_encode': (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    'msmd_audio_normalize': (_i, [_vp, _vp, _i, _i64, _vp]),
    'msmd_resample_linear': (_i, [_vp, _vp, _i, _i, _i, _vp]),
    'msmd_sample_window_ex': (_i, [_vp, _vp, _vp, C.c_uint64, _i, C.c_float, C.c_float, C.c_float, _i, _i, _vp, _vp, _vp, _vp]),
    'msmd_sample_window_sched': (_i, [_vp, _vp, _vp, C.c_uint64, _i, C.c_float, C.c_float, C.c_float, _i, _i, _vp, _vp, _vp,
                                      _vp, _vp]),
    'msmd_flame_create': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, C.POINTER(_vp)]),
    'msmd_flame_decode': (_i, [_vp, _vp, _vp, _i, _i64, _vp, _vp, _i, _vp]),
    'msmd_flame_destroy': (None, [_vp]),
    'msmd_vertices2landmarks': (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _vp]),
    'msmd_flame_contour_index': (_i, [_vp, _i, _i, _vp, _i, _i64, _vp, _vp]),
}

_lib = None


class MsmdError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MsmdError(f'{LIB_PATH} not found: build it with `python build.py` '
                            '(no CPU fallback exists for this package)')
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError if the export is missing: fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().msmd_last_error().decode()
        if rc == -1:
            raise ValueError(msg)
        raise MsmdError(f'msmd_b200 error {rc}: {msg}')


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dev_ptr(t, dtype=torch.float32, name='tensor'):
    """Device pointer of a contiguous CUDA tensor of the given dtype (raises otherwise)."""
    if t is None:
        return C.c_void_p(0)
    if not t.is_cuda:
        raise MsmdError(f'{name} must be a CUDA tensor: msmd_b200 has no CPU path')
    if t.dtype != dtype:
        raise TypeError(f'{name} must be {dtype}, got {t.dtype}')
    if not t.is_contiguous():
        raise ValueError(f'{name} must be contiguous')
    return C.c_void_p(t.data_ptr())


def as_f32c(t):
    """contiguous fp32 view/copy on the tensor's own (CUDA) device"""
    if not t.is_cuda:
        raise MsmdError('msmd_b200 has no CPU path: pass CUDA tensors')
    return t.to(torch.float32).contiguous()


def profile_query(name):
    """(total_ms, launches) of one instrumented kernel class since the last reset."""
    ms, n = C.c_double(0), C.c_int64(0)
    check(lib().msmd_profile_query(name.encode(), C.byref(ms), C.byref(n)))
    return ms.value, n.value


def profile_dump():
    """{kernel class: (total_ms, launches)} since the last reset."""
    buf = C.create_string_buffer(1 << 16)
    check(lib().msmd_profile_dump(buf, len(buf)))
    out = {}
    for line in buf.value.decode().splitlines():
        name, ms, n = line.rsplit(' ', 2)
        out[name] = (float(ms), int(n))
    return out
