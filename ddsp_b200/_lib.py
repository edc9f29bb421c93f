"""ctypes binding of libddsp_b200.so (the C ABI in include/ddsp_b200.h).

There is NO fallback: if the shared library is missing or fails to load, every
op raises.  Build it with `python -m ddsp_b200.build` (needs nvcc, not a GPU).
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libddsp_b200.so')

OK = 0
E_INVALID = -1
E_UNSUPPORTED = -2
E_CUDA = -3
E_WORKSPACE = -4

AMP_WINDOW = 0
AMP_LINEAR = 1
PHASE_RECURRENCE = 0
PHASE_DIRECT = 1
CTL_SCALE = 1
CTL_NYQUIST = 2
PAD_SAME = 0
PAD_VALID = 1
LTI_REVERSE_AUDIO = 1
LTI_REVERSE_IR = 2

_c_float_p = ctypes.c_void_p  # device pointers travel as integers
_i = ctypes.c_int
_i64 = ctypes.c_int64
_u64 = ctypes.c_uint64
_f = ctypes.c_float
_vp = ctypes.c_void_p
_sz = ctypes.c_size_t
_d = ctypes.c_double

# name -> (restype, argtypes); mirrors include/ddsp_b200.h one to one.
SIGNATURES = {
    'ddsp_b200_version': (_i, []),
    'ddsp_b200_last_error': (ctypes.c_char_p, []),
    'ddsp_b200_launch_count': (_u64, []),
    'ddsp_b200_harmonic_controls':
        (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _i, _vp]),
    'ddsp_b200_harmonic_forward':
        (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _i, _i, _vp]),
    'ddsp_b200_streaming_harmonic_forward':
        (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _vp]),
    'ddsp_b200_noise_controls': (_i, [_vp, _vp, _i64, _f, _i, _vp]),
    'ddsp_b200_ir_size': (_i, [_i, _i]),
    'ddsp_b200_frequency_impulse_response':
        (_i, [_vp, _vp, _i64, _i, _i, _vp]),
    'ddsp_b200_fir_time_varying':
        (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    'ddsp_b200_uniform_noise': (_i, [_vp, _i, _i, _u64, _u64, _vp]),
    'ddsp_b200_filtered_noise_workspace': (_sz, [_i, _i, _i, _i, _i]),
    'ddsp_b200_filtered_noise_forward':
        (_i, [_vp, _vp, _u64, _u64, _vp, _i, _i, _i, _i, _i, _i, _vp, _sz,
              _vp]),
    'ddsp_b200_decoder_forward':
        (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _u64, _vp, _i, _i, _i, _i, _i, _f,
              _i, _i, _i, _f, _vp]),
    'ddsp_b200_host_pipeline_create':
        (_i, [ctypes.POINTER(_vp), _i, _i, _i, _i, _i, _i]),
    'ddsp_b200_host_pipeline_destroy': (_i, [_vp]),
    'ddsp_b200_decoder_forward_host':
        (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _u64, _vp, _i, _i, _f, _i, _i, _i,
              _f, _vp]),
    'ddsp_b200_harmonic_backward':
        (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _vp]),
    'ddsp_b200_harmonic_backward_f0':
        (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _vp, _sz, _vp]),
    'ddsp_b200_harmonic_controls_backward':
        (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _i, _vp]),
    'ddsp_b200_noise_controls_backward': (_i, [_vp, _vp, _vp, _i64, _f, _vp]),
    'ddsp_b200_filtered_noise_backward':
        (_i, [_vp, _vp, _u64, _u64, _vp, _i, _i, _i, _i, _i, _vp]),
    'ddsp_b200_oscillator_bank_workspace': (_sz, [_i, _i, _i]),
    'ddsp_b200_oscillator_bank':
        (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _i, _vp, _sz, _vp]),
    'ddsp_b200_resample': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    'ddsp_b200_fft_convolve_lti_workspace': (_sz, [_i, _i, _i, _i]),
    'ddsp_b200_fft_convolve_lti':
        (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    'ddsp_b200_angular_cumsum':
        (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    'ddsp_b200_oscillator_bank_tf_sequential':
        (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _i, _i, _vp]),
    'ddsp_b200_sinusoidal_workspace': (_sz, [_i, _i, _i]),
    'ddsp_b200_sinusoidal_forward':
        (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _i, _vp, _sz, _vp]),
    'ddsp_b200_wavetable_workspace': (_sz, [_i, _i, _i, _i, _i, _i]),
    'ddsp_b200_wavetable_forward':
        (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _i, _vp, _sz, _vp]),
    'ddsp_b200_wavetable_backward':
        (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _vp, _sz,
              _vp]),
    'ddsp_b200_linear_lookup': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'ddsp_b200_mod_delay_workspace': (_sz, [_i, _i, _i]),
    'ddsp_b200_mod_delay_forward':
        (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _d, _d, _i, _i, _vp]),
    'ddsp_b200_mod_delay_backward':
        (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _d, _d, _i, _i, _vp, _sz,
              _vp]),
    'ddsp_b200_sigmoid': (_i, [_vp, _vp, _i64, _vp]),
    'ddsp_b200_add': (_i, [_vp, _vp, _vp, _i64, _vp]),
    'ddsp_b200_frame_window': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    'ddsp_b200_frame_window_adjoint':
        (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    'ddsp_b200_spectral_l1': (_i, [_vp, _vp, _vp, _vp, _i64, _f, _f, _i, _i, _vp]),
}

_lib = None
_lock = threading.Lock()


def load():
  """Loads the library once; raises RuntimeError loudly if it is absent."""
  global _lib
  if _lib is not None:
    return _lib
  with _lock:
    if _lib is not None:
      return _lib
    if not os.path.exists(LIB_PATH):
      raise RuntimeError(
          'ddsp_b200: %s is missing. The CUDA extension is the product - '
          'there is no CPU fallback. Build it with `python -m ddsp_b200.build` '
          '(or __graft_entry__.build()).' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
      fn = getattr(lib, name)  # AttributeError if the .so lacks a symbol
      fn.restype = restype
      fn.argtypes = argtypes
    _lib = lib
  return _lib


def check(rc):
  """Maps a C status to the reference's Python error convention."""
  if rc == OK:
    return
  msg = load().ddsp_b200_last_error().decode('utf-8', 'replace')
  if rc == E_INVALID:
    raise ValueError(msg)
  if rc == E_UNSUPPORTED:
    raise NotImplementedError(msg)
  raise RuntimeError('ddsp_b200 (status %d): %s' % (rc, msg))
