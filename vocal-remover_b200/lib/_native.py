"""ctypes binding of libvr_b200.so (C ABI declared in include/vr_b200.h).

There is deliberately NO fallback: if the CUDA library is missing or no GPU is visible the import /
context creation raises, it never routes through PyTorch or a CPU implementation.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('VR_LIB_PATH', os.path.join(os.path.dirname(_HERE), 'libvr_b200.so'))

c_i32, c_i64, c_vp, c_fp = ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p


class VrConfig(ctypes.Structure):
    _fields_ = [('device', c_i32), ('n_fft', c_i32), ('hop_length', c_i32), ('nout', c_i32),
                ('nout_lstm', c_i32), ('cropsize', c_i32), ('max_batch', c_i32), ('conv_mode', c_i32)]


# name -> (restype, argtypes); must stay in sync with include/vr_b200.h (tests/test_abi.py checks the names)
SIGNATURES = {
    'vr_create': (c_i32, [ctypes.POINTER(VrConfig), ctypes.POINTER(c_vp)]),
    'vr_destroy': (None, [c_vp]),
    'vr_last_error': (ctypes.c_char_p, [c_vp]),
    'vr_load_tensor': (c_i32, [c_vp, ctypes.c_char_p, c_i32, c_i32, ctypes.POINTER(c_i64), c_vp]),
    'vr_finalize_weights': (c_i32, [c_vp]),
    'vr_stft': (c_i32, [c_vp, c_fp, c_i64, c_vp, c_i64, c_fp, c_vp]),
    'vr_istft': (c_i32, [c_vp, c_vp, c_i64, c_fp, c_vp]),
    'vr_resample': (c_i32, [c_vp, c_fp, c_i32, c_i64, c_fp, c_i64, ctypes.c_double, c_vp, c_vp, c_i32, c_i32, c_vp]),
    'vr_predict_mask': (c_i32, [c_vp, c_fp, c_i32, c_fp, c_vp]),
    'vr_forward': (c_i32, [c_vp, c_fp, c_i32, c_fp, c_vp]),
    'vr_normaliser': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_fp, c_vp]),
    'vr_separate_windows': (c_i32, [c_vp, c_vp, c_i64, c_fp, c_i32, c_i32, c_i32, c_fp, c_i64, c_i64, c_i32, c_vp]),
    'vr_separate': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_fp, c_vp]),
    'vr_apply_mask': (c_i32, [c_vp, c_vp, c_fp, c_i64, c_vp, c_vp, c_vp]),
    'vr_mask_frame_min': (c_i32, [c_vp, c_fp, c_i64, c_fp, c_vp]),
    'vr_mask_apply_weight': (c_i32, [c_vp, c_fp, c_i64, c_fp, c_vp]),
    'vr_apply_mask_istft': (c_i32, [c_vp, c_vp, c_fp, c_i64, c_fp, c_fp, c_vp]),
    'vr_stft_range': (c_i32, [c_vp, c_fp, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp]),
    'vr_normaliser_range': (c_i32, [c_vp, c_vp, c_i64, c_i64, c_i64, c_fp, c_vp]),
    'vr_apply_mask_istft_range': (c_i32, [c_vp, c_vp, c_fp, c_i64, c_i64, c_i64, c_fp, c_fp, c_vp]),
    'vr_separate_wave': (c_i32, [c_vp, c_fp, c_i64, c_i32, c_fp, c_fp, c_vp]),
    'vr_separate_wave_host': (c_i32, [c_vp, c_fp, c_i64, c_i32, c_fp, c_fp, c_vp]),
    'vr_separate_many': (c_i32, [c_vp, c_i32, ctypes.POINTER(c_vp), ctypes.POINTER(c_i64), c_i32,
                                 ctypes.POINTER(c_vp), c_vp]),
    'vr_separate_waves': (c_i32, [c_vp, c_i32, ctypes.POINTER(c_vp), ctypes.POINTER(c_i64), c_i32,
                                  ctypes.POINTER(c_vp), ctypes.POINTER(c_vp), c_vp]),
    'vr_shared_alloc': (c_i32, [c_vp, c_i64, ctypes.POINTER(c_vp), ctypes.c_char_p]),
    'vr_shared_open': (c_i32, [c_vp, ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    'vr_shared_close': (c_i32, [c_vp, c_vp, c_i32]),
    'vr_launch_count': (c_i64, [c_vp]),
    'vr_profile_enable': (c_i32, [c_vp, c_i32]),
    'vr_profile_read': (c_i32, [c_vp, ctypes.POINTER(ctypes.c_double)]),
    'vr_profile_dump': (c_i32, [c_vp, ctypes.c_char_p, c_i64, ctypes.POINTER(c_i64)]),
    'vr_debug_conv': (c_i32, [c_vp, c_fp, c_i32, c_i32, c_i32, c_i32, c_fp, c_fp, c_i32, c_i32, c_i32, c_i32, c_i32,
                              c_i32, c_i32, c_fp, c_vp]),
    'vr_debug_decoder': (c_i32, [c_vp, c_fp, c_i32, c_i32, c_i32, c_i32, c_fp, c_i32, c_fp, c_fp, c_i32, c_i32, c_i32,
                                 c_fp, c_vp]),
    'vr_debug_set': (c_i32, [c_i32, c_i32]),
    'vr_debug_trace': (c_i64, [c_vp, c_i64]),
    'vr_debug_read': (c_i32, [c_vp, ctypes.c_char_p, c_fp, c_i64, ctypes.POINTER(c_i64), c_vp]),
}

_lib = None


def load_library():
    """Loads libvr_b200.so; raises (loudly) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'libvr_b200.so not found at %s: build it with `python vocal-remover_b200/build.py` '
            '(or __graft_entry__.build()). There is no CPU / PyTorch fallback for the hot path.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the ABI is out of sync
        fn.restype = res
        fn.argtypes = args
    # validation knobs of the tensor-core kernels (see vr_debug_set in include/vr_b200.h)
    if os.environ.get('VR_FUSE_UP'):
        lib.vr_debug_set(5, int(os.environ['VR_FUSE_UP']))
    if os.environ.get('VR_KSKIP'):
        lib.vr_debug_set(6, int(os.environ['VR_KSKIP']))
    if os.environ.get('VR_USLOTS'):
        lib.vr_debug_set(4, int(os.environ['VR_USLOTS']))
    if os.environ.get('VR_NO_ROWS'):
        lib.vr_debug_set(1, int(os.environ['VR_NO_ROWS']))
    _lib = lib
    return lib


class NativeError(RuntimeError):
    pass


class Context(object):
    """One vr_ctx: a CascadedNet bound to one GPU, a cropsize and a maximum window batch."""

    def __init__(self, device_index, n_fft, hop_length, nout, nout_lstm, cropsize, max_batch, conv_mode=0):
        self.lib = load_library()
        self.cfg = VrConfig(int(device_index), int(n_fft), int(hop_length), int(nout), int(nout_lstm),
                            int(cropsize), int(max_batch), int(conv_mode))
        h = c_vp()
        rc = self.lib.vr_create(ctypes.byref(self.cfg), ctypes.byref(h))
        if rc != 0:
            raise NativeError('vr_create failed: %s' % self.lib.vr_last_error(None).decode())
        self.handle = h
        self.device_index = int(device_index)

    def close(self):
        if getattr(self, 'handle', None):
            self.lib.vr_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc, what):
        if rc != 0:
            raise NativeError('%s failed: %s' % (what, self.lib.vr_last_error(self.handle).decode()))

    def load_state_dict(self, sd):
        """sd: mapping key -> torch tensor or numpy array (the reference checkpoint format, SURVEY App. C)."""
        for key, val in sd.items():
            arr = val.detach().cpu().numpy() if hasattr(val, 'detach') else np.asarray(val)
            if arr.dtype == np.int64:
                dtype = 1
            else:
                arr = arr.astype(np.float32, copy=False)
                dtype = 0
            if not arr.flags.c_contiguous:
                arr = arr.copy(order='C')
            shape = (c_i64 * max(1, arr.ndim))(*arr.shape)
            self.check(self.lib.vr_load_tensor(self.handle, key.encode(), dtype, arr.ndim, shape,
                                               arr.ctypes.data_as(c_vp)), 'vr_load_tensor(%s)' % key)
        self.check(self.lib.vr_finalize_weights(self.handle), 'vr_finalize_weights')

    def launch_count(self):
        return int(self.lib.vr_launch_count(self.handle))


def stream_ptr():
    import torch
    return c_vp(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return c_vp(t.data_ptr())


def ptr_array(tensors):
    """HOST array of the tensors' device pointers (None gives NULL), as vr_separate_many / vr_separate_waves take."""
    return (c_vp * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def i64_array(values):
    return (c_i64 * len(values))(*[int(v) for v in values])
