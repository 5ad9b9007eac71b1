"""ctypes binding of libmpa.so (the C ABI declared in include/mpa.h).

There is deliberately no fallback: if the shared library is missing or the device is not sm_100 every
operator raises.  PyTorch is used for device memory and streams only."""
import ctypes
import os
import re

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libmpa.so')
HEADER_PATH = os.path.join(os.path.dirname(_HERE), 'include', 'mpa.h')

_lib = None


class MpaError(RuntimeError):
    pass


def declared_symbols():
    """Every function name declared in include/mpa.h (used by the symbol-export test)."""
    src = open(HEADER_PATH).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(mpa_[a-z0-9_]+)\s*\(', src)))


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MpaError(f'{LIB_PATH} is missing: build it with `python -m multipitch_architectures_b200.build` '
                           '(nvcc, sm_100a).  There is no CPU / PyTorch fallback.')
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.mpa_last_error.restype = ctypes.c_char_p
        _lib.mpa_launch_count.restype = ctypes.c_longlong
        for name in ('mpa_encoder_layer_workspace', 'mpa_conv_tc_packed_bytes', 'mpa_conv_tc_packed_bytes_fmt', 'mpa_conv_tc_pool_workspace_fmt', 'mpa_tuning_workspace', 'mpa_cqt_levels_bwd_workspace', 'mpa_conv_tc_pool_workspace', 'mpa_conv_tc_ring_packed_bytes', 'mpa_gemm_tc_chunked_bytes', 'mpa_eval_workspace', 'mpa_lstm_layer_workspace', 'mpa_lstm_layer_bwd_workspace', 'mpa_conv_rows_fwd_workspace'):
            if hasattr(_lib, name):
                getattr(_lib, name).restype = ctypes.c_size_t
    return _lib


def last_error():
    return lib().mpa_last_error().decode()


def launch_count():
    return int(lib().mpa_launch_count())


def _conv(a):
    if isinstance(a, torch.Tensor):
        if not a.is_cuda:
            raise MpaError('libmpa operators take CUDA tensors only (no CPU path exists)')
        if not a.is_contiguous():
            raise MpaError('libmpa operators take contiguous tensors')
        if a.device.index != torch.cuda.current_device():
            # the launch goes to the CURRENT device's stream: a tensor of another GPU would fault with an illegal address
            raise MpaError(f'tensor lives on cuda:{a.device.index} but the current device is cuda:{torch.cuda.current_device()}: '
                           'wrap the call in `with torch.cuda.device(...)`')
        return ctypes.c_void_p(a.data_ptr())
    if a is None:
        return ctypes.c_void_p(0)
    if isinstance(a, float):
        return ctypes.c_float(a)
    if isinstance(a, bool):
        return ctypes.c_int(int(a))
    if isinstance(a, int):
        return ctypes.c_int(a)
    return a


def call(name, *args):
    """Invoke `int mpa_<name>(...)`; tensors -> device pointers, float -> c_float, int -> c_int.
    Pass ctypes values explicitly for long long / size_t parameters."""
    fn = getattr(lib(), 'mpa_' + name)
    rc = fn(*[_conv(a) for a in args])
    if rc != 0:
        raise MpaError(f'mpa_{name} failed ({rc}): {last_error()}')


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def i64(v):
    return ctypes.c_longlong(int(v))


def usize(v):
    return ctypes.c_size_t(int(v))


def u64(v):
    return ctypes.c_ulonglong(int(v) & 0xFFFFFFFFFFFFFFFF)
