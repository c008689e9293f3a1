"""
ctypes binding of librepet_b200.so (include/repet_b200.h) and the host-side parameter
derivation of the REPET drivers.

This is the reference-side binding of INTEGRATION.md: every derived integer is computed with
the reference's own Python expression (cited per line), the samples go to the library
untouched, and there is NO CPU fallback -- if the CUDA library or a CUDA device is missing
the calls raise.
"""

import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "librepet_b200.so")

REPET_OK = 0
REPET_E_INVALID_ARG = -1
REPET_E_TOO_SHORT = -2
REPET_E_CUDA = -3
REPET_E_OOM = -4
REPET_E_UNSUPPORTED = -5


class RepetParams(ctypes.Structure):
    """struct repet_params of include/repet_b200.h."""

    _fields_ = [
        ("window_length", ctypes.c_int32),
        ("step_length", ctypes.c_int32),
        ("period_lo", ctypes.c_int32),
        ("period_hi", ctypes.c_int32),
        ("cutoff_bins", ctypes.c_int32),
        ("segment_length", ctypes.c_int32),
        ("segment_step", ctypes.c_int32),
        ("filter_order", ctypes.c_int32),
        ("similarity_distance", ctypes.c_int32),
        ("similarity_number", ctypes.c_int32),
        ("buffer_frames", ctypes.c_int32),
        ("online_frame_base", ctypes.c_int32),
        ("similarity_threshold", ctypes.c_double),
        ("cola_gain", ctypes.c_double),
    ]


_lib = None
_lib_lock = threading.Lock()

_c_int = ctypes.c_int
_c_i64 = ctypes.c_int64
_c_u64 = ctypes.c_uint64
_vp = ctypes.c_void_p
_pp = ctypes.POINTER(RepetParams)

# name -> (restype, argtypes); must list every symbol include/repet_b200.h declares
SIGNATURES = {
    "repet_version": (ctypes.c_char_p, []),
    "repet_create": (_c_int, [_c_int, ctypes.POINTER(_vp)]),
    "repet_destroy": (_c_int, [_vp]),
    "repet_last_error": (ctypes.c_char_p, [_vp]),
    "repet_set_stream": (_c_int, [_vp, _vp]),
    "repet_set_window": (_c_int, [_vp, _vp, _c_int]),
    "repet_set_workspace_limit": (_c_int, [_vp, _c_u64]),
    "repet_workspace_bytes": (_c_u64, [_vp]),
    "repet_synchronize": (_c_int, [_vp]),
    "repet_launch_count": (_c_u64, [_vp]),
    "repet_set_tuning": (_c_int, [ctypes.c_char_p, _c_int]),
    "repet_set_profiling": (_c_int, [_vp, _c_int]),
    "repet_profile_read": (_c_int, [_vp, _vp, _vp, _c_int]),
    "repet_kernel_name": (ctypes.c_char_p, [_c_int]),
    "repet_original_batch_dev": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp, _vp]),
    "repet_original_batch": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp]),
    "repet_original_batch_pcm16": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp]),
    "repet_separate_batch": (_c_int, [_vp, _c_int, _vp, _c_int, _c_int, _c_int, _c_i64, _pp, _vp, _c_int, _vp]),
    "repet_ints_per_clip": (_c_i64, [_c_int, _pp, _c_i64]),
    "repet_host_alloc": (_c_int, [ctypes.POINTER(_vp), _c_u64]),
    "repet_host_free": (_c_int, [_vp]),
    "repet_host_register": (_c_int, [_vp, _c_u64]),
    "repet_host_unregister": (_c_int, [_vp]),
    "repet_device_count": (_c_int, []),
    "repet_original_f64": (_c_int, [_vp, _vp, _c_i64, _c_int, _pp, _vp, _vp]),
    "repet_extended_segments": (_c_int, [_pp, _c_i64]),
    "repet_extended_batch_dev": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp, _vp]),
    "repet_extended_batch": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp]),
    "repet_extended_f64": (_c_int, [_vp, _vp, _c_i64, _c_int, _pp, _vp, _vp, _c_int]),
    "repet_adaptive_batch_dev": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp, _vp]),
    "repet_adaptive_batch": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp]),
    "repet_adaptive_f64": (_c_int, [_vp, _vp, _c_i64, _c_int, _pp, _vp, _vp, _c_int]),
    "repet_adaptivemask": (_c_int, [_vp, _vp, _c_int, _vp, _c_int, _vp]),
    "repet_beatspectrogram": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp]),
    "repet_selfsimilarity": (_c_int, [_vp, _vp, _c_int, _c_int, _vp]),
    "repet_similarity": (_c_int, [_vp, _vp, _c_int, _vp, _c_int, _c_int, _vp]),
    "repet_localmaxima": (_c_int, [_vp, _vp, _c_int, _c_int, ctypes.c_double, _c_int, _c_int, _vp, _vp, _vp]),
    "repet_simmask": (_c_int, [_vp, _vp, _c_int, _vp, _vp, _c_int, _vp]),
    "repet_acorr": (_c_int, [_vp, _vp, _c_int, _c_int, _vp]),
    "repet_periods": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp]),
    "repet_sim_batch_dev": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp, _vp]),
    "repet_sim_batch": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp]),
    "repet_sim_f64": (_c_int, [_vp, _vp, _c_i64, _c_int, _pp, _vp, _vp, _c_int]),
    "repet_simonline_frames": (_c_int, [_pp, _c_i64]),
    "repet_simonline_batch_dev": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp, _vp]),
    "repet_simonline_batch": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp, _vp]),
    "repet_simonline_f64": (_c_int, [_vp, _vp, _c_i64, _c_int, _pp, _vp, _vp, _c_int]),
    "repet_simonline_open": (_c_int, [_vp, _pp, _c_int, ctypes.POINTER(_vp)]),
    "repet_simonline_block": (_c_int, [_vp, _vp, _c_i64, _vp, _c_i64, ctypes.POINTER(_c_i64)]),
    "repet_simonline_flush": (_c_int, [_vp, _vp, _c_i64, ctypes.POINTER(_c_i64)]),
    "repet_simonline_close": (_c_int, [_vp]),
    "repet_separate_f64": (_c_int, [_vp, _c_int, _vp, _c_i64, _c_int, _pp, _vp, _vp, _vp, _vp, _c_int]),
    "repet_spectrogram_pitch": (_c_int, [_pp]),
    "repet_spectrogram_frames": (_c_int, [_pp, _c_i64]),
    "repet_spectrogram_batch_dev": (_c_int, [_vp, _vp, _c_int, _c_int, _c_i64, _pp, _vp]),
    "repet_foreground_dev": (_c_int, [_vp, _vp, _vp, _c_i64, _vp]),
    "repet_general_f64": (_c_int, [_vp, _c_int, _vp, _c_i64, _c_int, _pp, _vp, _vp, _vp, _c_i64]),
    "repet_stft_frames": (_c_int, [_c_i64, _c_int, _c_int]),
    "repet_stft_f64": (_c_int, [_vp, _vp, _c_i64, _vp, _c_int, _c_int, _vp, _vp]),
    "repet_istft_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _vp, _c_int, _vp, ctypes.POINTER(_c_i64)]),
    "repet_acorr_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _vp]),
    "repet_beatspectrum_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _vp]),
    "repet_stft": (_c_int, [_vp, _vp, _c_int, _c_i64, _vp, _vp, _vp]),
    "repet_istft": (_c_int, [_vp, _vp, _c_int, _c_int, ctypes.c_double, _vp]),
    "repet_beatspectrum": (_c_int, [_vp, _vp, _c_int, _c_int, _vp]),
    "repet_period": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp]),
    "repet_mask": (_c_int, [_vp, _vp, _c_int, _c_int, _vp]),
}


def load_library():
    """Load librepet_b200.so; raises if it has not been built (python repet-python_b200/build.py)."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise ImportError(
                "librepet_b200.so is missing at %s -- build it with `python repet-python_b200/build.py`; "
                "there is no CPU fallback" % LIB_PATH
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
        return lib


class RepetError(RuntimeError):
    pass


def _ptr(array):
    return array.ctypes.data_as(_vp) if array is not None else None


class Handle:
    """One library handle (one GPU, one host thread)."""

    def __init__(self, device=0):
        self.lib = load_library()
        handle = _vp()
        rc = self.lib.repet_create(int(device), ctypes.byref(handle))
        if rc != REPET_OK:
            raise RepetError(
                "repet_create(device=%d) failed with status %d: no usable CUDA device (there is no CPU fallback)"
                % (device, rc)
            )
        self.h = handle
        self.device = int(device)
        self._window_key = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.repet_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc == REPET_OK:
            return
        message = self.lib.repet_last_error(self.h).decode("utf-8", "replace")
        if rc in (REPET_E_INVALID_ARG, REPET_E_TOO_SHORT):
            raise ValueError(message)  # what NumPy raises inside the reference (quirk Q17)
        if rc == REPET_E_UNSUPPORTED:
            raise NotImplementedError(message)
        if rc == REPET_E_OOM:
            raise MemoryError(message)
        raise RepetError("status %d: %s" % (rc, message))

    def set_window(self, window_function, key=None):
        window = np.ascontiguousarray(window_function, dtype=np.float64)
        self.check(self.lib.repet_set_window(self.h, _ptr(window), len(window)))
        self._window_key = key

    def ensure_window(self, window_length):
        """Upload the drivers' periodic Hamming window unless it is already the current one."""
        if self._window_key != ("hamming", window_length):
            self.set_window(hamming_window(window_length), key=("hamming", window_length))

    def set_stream(self, cuda_stream_pointer):
        """Enqueue on an existing CUDA stream (e.g. torch.cuda.current_stream().cuda_stream).
        None restores the handle's own stream; 0 means the legacy default stream, which the
        runtime spells cudaStreamLegacy = 0x1."""
        if cuda_stream_pointer is None:
            pointer = None
        else:
            pointer = _vp(int(cuda_stream_pointer) or 1)
        self.check(self.lib.repet_set_stream(self.h, pointer))

    def set_workspace_limit(self, number_bytes):
        self.check(self.lib.repet_set_workspace_limit(self.h, int(number_bytes)))

    def workspace_bytes(self):
        """Bytes of device workspace the handle holds (grown on demand, kept between calls)."""
        return int(self.lib.repet_workspace_bytes(self.h))

    def synchronize(self):
        self.check(self.lib.repet_synchronize(self.h))

    def launch_count(self):
        return int(self.lib.repet_launch_count(self.h))

    def set_profiling(self, on):
        self.check(self.lib.repet_set_profiling(self.h, 1 if on else 0))

    def profile_read(self, reset=True):
        """{kernel name: (total ms, launches)} accumulated while profiling was on."""
        ms = np.zeros(12, dtype=np.float64)
        counts = np.zeros(12, dtype=np.uint64)
        self.check(self.lib.repet_profile_read(self.h, _ptr(ms), _ptr(counts), 1 if reset else 0))
        return {
            self.lib.repet_kernel_name(i).decode(): (float(ms[i]), int(counts[i])) for i in range(12) if counts[i]
        }


def set_tuning(**knobs):
    """Process-wide launch-shape knobs (see repet_set_tuning in include/repet_b200.h)."""
    lib = load_library()
    for name, value in knobs.items():
        if lib.repet_set_tuning(name.encode(), int(value)) != REPET_OK:
            raise ValueError("unknown tuning knob %r" % name)


_handles = {}


def get_handle(device=None):
    """Process-wide handle of a device (default: REPET_DEVICE or LOCAL_RANK or 0)."""
    if device is None:
        device = int(os.environ.get("REPET_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    if device not in _handles:
        _handles[device] = Handle(device)
    return _handles[device]


# ------------------------------------------------------------------------------------------
# parameter derivation, with the reference's own expressions
# ------------------------------------------------------------------------------------------
def hamming_window(window_length):
    """scipy.signal.hamming(N, sym=False) (repet.py:131); SciPy's own values, which differ
    from the closed form by up to 1 ulp."""
    import scipy.signal.windows

    return scipy.signal.windows.hamming(window_length, sym=False)


_PARAM_CACHE = {}


def derive_params(sampling_frequency, tunables, driver="original"):
    """Cached front end of _derive_params (the derivation is pure; batch callers hit it every step)."""
    try:
        # array-likes (lists, tuples, NumPy arrays -- the reference takes np.array(period_range)) become tuples,
        # NumPy scalars plain numbers
        key = (float(sampling_frequency), driver,
               tuple((k, tuple(np.ravel(v).tolist()) if np.ndim(v) else (v.item() if isinstance(v, np.generic) else v))
                     for k, v in sorted(tunables.items())))
        hit = _PARAM_CACHE.get(key)
    except TypeError:  # an unhashable tunable: derive uncached
        key, hit = None, None
    if hit is None:
        hit = _derive_params(sampling_frequency, tunables, driver)
        if key is not None:
            if len(_PARAM_CACHE) > 64:
                _PARAM_CACHE.clear()
            _PARAM_CACHE[key] = hit
    params = RepetParams()
    ctypes.memmove(ctypes.byref(params), ctypes.byref(hit[0]), ctypes.sizeof(RepetParams))
    return params, hit[1]


def _derive_params(sampling_frequency, tunables, driver="original"):
    """All derived integers of the five drivers (SURVEY.md quirk Q16).  `driver` selects the
    unit of the segment sizes: samples for extended (repet.py:266-267), frames for adaptive
    (repet.py:519-520)."""
    window_length = pow(2, int(np.ceil(np.log2(0.04 * sampling_frequency))))  # repet.py:130
    step_length = int(window_length / 2)  # repet.py:132
    window_function = hamming_window(window_length)
    period_range2 = np.round(np.array(tunables["period_range"]) * sampling_frequency / step_length).astype(int)  # :165
    cutoff_frequency2 = round(tunables["cutoff_frequency"] * window_length / sampling_frequency)  # :173
    p = RepetParams()
    p.window_length = window_length
    p.step_length = step_length
    p.period_lo = int(period_range2[0])
    p.period_hi = int(period_range2[1])
    p.cutoff_bins = int(cutoff_frequency2)
    p.filter_order = int(tunables["filter_order"])
    p.similarity_distance = int(round(tunables["similarity_distance"] * sampling_frequency / step_length))  # :670
    p.similarity_number = int(tunables["similarity_number"])
    p.similarity_threshold = float(tunables["similarity_threshold"])
    p.buffer_frames = int(round((tunables["buffer_length"] * sampling_frequency) / step_length))  # :787
    p.cola_gain = float(sum(window_function[0:window_length:step_length]))  # repet.py:1103
    if driver == "extended":
        p.segment_length = round(tunables["segment_length"] * sampling_frequency)  # repet.py:266
        p.segment_step = round(tunables["segment_step"] * sampling_frequency)  # repet.py:267
    else:
        p.segment_length = int(round(tunables["segment_length"] * sampling_frequency / step_length))  # repet.py:519
        p.segment_step = int(round(tunables["segment_step"] * sampling_frequency / step_length))  # repet.py:520
    return p, window_function


def number_of_frames(number_samples, window_length, step_length):
    """repet.py:135-146."""
    return int(np.ceil(((number_samples + 2 * int(np.floor(window_length / 2))) - window_length) / step_length)) + 1


# ------------------------------------------------------------------------------------------
# drivers
# ------------------------------------------------------------------------------------------
FAST_WINDOWS = (512, 1024, 2048)  # window lengths of the register-blocked fp32 frame transforms
METHODS = {"original": 0, "extended": 1, "adaptive": 2, "sim": 3, "simonline": 4}
FORMATS = {"f32": 0, "pcm16": 1}  # REPET_FMT_F32_PLANAR, REPET_FMT_PCM16
SPECTROGRAMS = ("audio_spectrogram", "background_spectrogram", "foreground_spectrogram")


def needs_general_path(params, number_channels):
    """Inputs the fast fp32 kernels are not compiled for: sampling rates above 51.2 kHz (window 4096 at 96 kHz, 8192
    at 192 kHz, repet.py:130) and more than two channels.  They run on the general float64 device path
    (repet_general_f64); so does anything else the fast path answers with REPET_E_UNSUPPORTED (period ranges above
    1024 frames, ...)."""
    return params.window_length not in FAST_WINDOWS or number_channels > 2


def _route(params, number_channels, fast, general):
    """The one rule between the two device paths: `fast()`, unless the fast kernels are not compiled for the input
    (needs_general_path) or refuse it (NotImplementedError, i.e. REPET_E_UNSUPPORTED: a period range above 1024
    frames, ...); then `general()`.  Every other error propagates."""
    if not needs_general_path(params, number_channels):
        try:
            return fast()
        except NotImplementedError:
            pass
    return general()


def _ints_per_clip(lib, method, params, number_samples):
    return int(lib.repet_ints_per_clip(METHODS[method], ctypes.byref(params), number_samples))


def _run_f64(method, audio_signal, params, window_function, handle=None, foreground=False, spectrograms=False):
    """One clip of `method`, float64 (samples, channels) in and out, on the path _route picks.  `params` and
    `window_function` come from derive_params (callers may set online_frame_base).  Returns a dict: background,
    integers (the method's integer output), and on request foreground and the three display spectrograms
    (SPECTROGRAMS, which need `foreground` too)."""
    _, number_channels = np.shape(audio_signal)  # ValueError if not 2-D, as in the reference
    handle = handle or get_handle()
    return _route(params, number_channels,
                  lambda: _fast_f64(method, audio_signal, params, handle, foreground, spectrograms),
                  lambda: _general_f64(method, audio_signal, params, window_function, handle, foreground, spectrograms))


def _fast_f64(method, audio_signal, params, handle, foreground=False, spectrograms=False):
    """The fast route of _run_f64 (repet_separate_f64) alone: raises NotImplementedError where the fast kernels
    refuse the input.  The foreground and the spectrograms are formed on the device from the buffers already there."""
    audio = np.ascontiguousarray(audio_signal, dtype=np.float64)
    number_samples, number_channels = audio.shape
    lib = handle.lib
    handle.ensure_window(params.window_length)
    capacity = _ints_per_clip(lib, method, params, number_samples)
    background = np.empty_like(audio)
    ints = np.zeros(max(1, capacity), dtype=np.int32)
    fg = np.empty_like(audio) if foreground else None
    spec = None
    if spectrograms:
        spec = np.empty((3, lib.repet_spectrogram_frames(ctypes.byref(params), number_samples),
                         lib.repet_spectrogram_pitch(ctypes.byref(params))), dtype=np.float32)
    handle.check(
        lib.repet_separate_f64(
            handle.h, METHODS[method], _ptr(audio), number_samples, number_channels, ctypes.byref(params),
            _ptr(background), _ptr(fg), _ptr(spec), _ptr(ints), len(ints),
        )
    )
    result = {"background": background}
    if foreground:
        result["foreground"] = fg
    result["integers"] = ints[:capacity]
    if spectrograms:
        number_frequencies = params.window_length // 2 + 1
        for i, name in enumerate(SPECTROGRAMS):
            result[name] = spec[i, :, :number_frequencies].T.astype(np.float64)
    return result


def _single_f64_fast(entry, driver, audio_signal, sampling_frequency, tunables, handle, ints_capacity):
    """The fast kernels alone through a per-driver entry point `entry` (repet_<driver>_f64, kept public for C
    integrators): no routing, so a refusal raises NotImplementedError.  For tests that need the fast kernels' own
    answer on that entry point; `ints_capacity(params, number_samples)` sizes the integer output."""
    number_samples, number_channels = np.shape(audio_signal)
    params, _ = derive_params(sampling_frequency, tunables, driver)
    handle.ensure_window(params.window_length)
    audio = np.ascontiguousarray(audio_signal, dtype=np.float64)
    background = np.empty((number_samples, number_channels), dtype=np.float64)
    capacity = ints_capacity(params, number_samples)
    ints = np.zeros(max(1, capacity), dtype=np.int32)
    handle.check(
        getattr(handle.lib, entry)(
            handle.h, _ptr(audio), number_samples, number_channels, ctypes.byref(params), _ptr(background), _ptr(ints),
            len(ints),
        )
    )
    return background, ints[:capacity]


def _general_f64(method, audio_signal, params, window_function, handle, foreground=False, spectrograms=False):
    """The general route of _run_f64 (repet_general_f64).  The foreground and the spectrograms are formed on the
    host from its outputs (foreground = audio - background, README.md:68; spectrograms by the general _stft,
    README.md:79-81)."""
    audio = np.ascontiguousarray(audio_signal, dtype=np.float64)
    number_samples, number_channels = audio.shape
    window = np.ascontiguousarray(window_function, dtype=np.float64)
    capacity = _ints_per_clip(handle.lib, method, params, number_samples)
    background = np.empty_like(audio)
    ints = np.zeros(max(1, capacity), dtype=np.int32)
    handle.check(
        handle.lib.repet_general_f64(
            handle.h, METHODS[method], _ptr(audio), number_samples, number_channels, ctypes.byref(params), _ptr(window),
            _ptr(background), _ptr(ints), len(ints),
        )
    )
    result = {"background": background}
    if foreground:
        result["foreground"] = audio - background
    result["integers"] = ints[:capacity]
    if spectrograms:
        half = params.window_length // 2 + 1
        for name, signal in zip(SPECTROGRAMS, (audio, background, result["foreground"])):
            result[name] = np.abs(stft_general(np.mean(signal, axis=1), window_function, params.step_length,
                                               handle=handle)[0:half, :])
    return result


def _run_batch(method, audio, params, window_function, handle=None, in_format="f32", out_format="f32", out=None,
               devices=None):
    """A batch of equally long clips of `method` in host memory, on the path _route picks: the fast kernels
    (repet_separate_batch, clip-sharded over `devices` when given; a refusal of any shard sends the whole batch to
    the general path), or clip by clip the general float64 path on the caller's handle.  Returns (background in
    `out_format`, integers (clips, max(1, per clip)) int32)."""
    in_code, out_code = FORMATS[in_format], FORMATS[out_format]
    audio = np.ascontiguousarray(audio, dtype=np.int16 if in_code else np.float32)
    if audio.ndim != 3:
        raise ValueError("audio must have shape (clips, channels, samples) [f32] or (clips, samples, channels) [pcm16]")
    if in_code:
        number_clips, number_samples, number_channels = audio.shape
    else:
        number_clips, number_channels, number_samples = audio.shape
    out_shape = (number_clips, number_samples, number_channels) if out_code else (number_clips, number_channels, number_samples)
    out_dtype = np.int16 if out_code else np.float32
    if out is None:
        out = np.empty(out_shape, dtype=out_dtype)
    elif out.shape != out_shape or out.dtype != out_dtype or not out.flags.c_contiguous:
        raise ValueError("out must be a C-contiguous %s array of shape %s" % (np.dtype(out_dtype).name, out_shape))
    if devices is not None:
        devices = [int(d) for d in devices]
    per_clip = _ints_per_clip(load_library(), method, params, number_samples)
    ints = np.zeros((number_clips, max(1, per_clip)), dtype=np.int32)

    def run(h, first, stop):
        if stop <= first:
            return
        h.ensure_window(params.window_length)
        h.check(h.lib.repet_separate_batch(
            h.h, METHODS[method], _ptr(audio[first:stop]), in_code, stop - first, number_channels, number_samples,
            ctypes.byref(params), _ptr(out[first:stop]), out_code, _ptr(ints[first:stop])))

    def fast():
        if devices is None:
            run(handle or get_handle(), 0, number_clips)
        else:
            shards = shard_bounds(number_clips, len(devices))
            _run_shards([(lambda h, lo=lo, hi=hi: run(h, lo, hi)) for lo, hi in shards], devices)
        return out, ints

    def general():
        h = handle or get_handle()
        for i, clip in enumerate(audio):
            x = clip / 32768.0 if in_code else clip.T  # repet.py:929
            result = _general_f64(method, x, params, window_function, h)
            y = result["background"]
            if out_code:
                out[i] = np.clip(np.rint(y.astype(np.float32) * np.float32(32768.0)), -32768, 32767).astype(np.int16)
            else:
                out[i] = y.T
            ints[i, : len(result["integers"])] = result["integers"]
        return out, ints

    return _route(params, number_channels, fast, general)


def general_f64(method, audio_signal, sampling_frequency, tunables, handle=None):
    """Any of the five drivers on the general float64 device path.  Returns (background float64 (S, C), ints int32)."""
    params, window_function = derive_params(sampling_frequency, tunables, method)
    result = _general_f64(method, audio_signal, params, window_function, handle or get_handle())
    return result["background"], result["integers"]


def original_f64(audio_signal, sampling_frequency, tunables, handle=None, return_period=False):
    """repet.original with the reference's calling convention (repet.py:67-202)."""
    params, window_function = derive_params(sampling_frequency, tunables)
    result = _run_f64("original", audio_signal, params, window_function, handle)
    if return_period:
        return result["background"], int(result["integers"][0])
    return result["background"]


def original_batch(audio, sampling_frequency, tunables, handle=None, out=None):
    """`original` over a batch of clips: audio (B, C, S) float32 planar, host memory.
    Returns (background (B, C, S) float32, periods (B,) int32)."""
    params, window_function = derive_params(sampling_frequency, tunables)
    background, ints = _run_batch("original", audio, params, window_function, handle, out=out)
    return background, ints[:, 0]


def original_batch_device(audio_ptr, background_ptr, number_clips, number_channels, number_samples,
                          sampling_frequency, tunables, handle=None, periods_ptr=None, periods_host=None):
    """`original` over device-resident fp32 planar clips (raw device pointers, e.g.
    torch.Tensor.data_ptr()).  Enqueues on the handle's stream; synchronises only when
    `periods_host` (int32 array) is given."""
    handle = handle or get_handle()
    params, _ = derive_params(sampling_frequency, tunables)
    handle.ensure_window(params.window_length)
    handle.check(
        handle.lib.repet_original_batch_dev(
            handle.h, _vp(audio_ptr), number_clips, number_channels, number_samples, ctypes.byref(params),
            _vp(background_ptr), _vp(periods_ptr) if periods_ptr else None, _ptr(periods_host),
        )
    )


# ------------------------------------------------------------------------------------------
# helpers with the reference's shapes
# ------------------------------------------------------------------------------------------
def stft_half(signals, window_function, step_length, handle=None, with_power=False):
    """Half spectra of 1 or 2 real signals: signals (C, S) -> complex64 (C, T, F) [, power (T, F)]."""
    handle = handle or get_handle()
    window_length = len(window_function)
    if step_length * 2 != window_length:
        raise NotImplementedError("step_length must be window_length/2")
    handle.set_window(window_function)
    signals = np.ascontiguousarray(signals, dtype=np.float32)
    number_channels, number_samples = signals.shape
    number_times = number_of_frames(number_samples, window_length, step_length)
    half = window_length // 2
    packed = np.empty((number_times, number_channels, half, 2), dtype=np.float32)
    power = np.empty((number_times, half + 1), dtype=np.float32) if with_power else None
    frames = ctypes.c_int32(0)
    handle.check(
        handle.lib.repet_stft(
            handle.h, _ptr(signals), number_channels, number_samples, _ptr(packed), _ptr(power), ctypes.byref(frames)
        )
    )
    assert frames.value == number_times
    spectrum = np.empty((number_channels, number_times, half + 1), dtype=np.complex64)
    body = packed[..., 0] + 1j * packed[..., 1]
    spectrum[:, :, :half] = np.transpose(body, (1, 0, 2))
    spectrum[:, :, 0] = packed[:, :, 0, 0].T  # DC is real
    spectrum[:, :, half] = packed[:, :, 0, 1].T  # Nyquist rides in bin 0's imaginary slot
    if with_power:
        return spectrum, power
    return spectrum


def istft_half(spectrum, window_function, step_length, handle=None):
    """Inverse of stft_half: complex (C, T, F) -> float32 (C, (T-1)*H)."""
    handle = handle or get_handle()
    window_length = len(window_function)
    if step_length * 2 != window_length:
        raise NotImplementedError("step_length must be window_length/2")
    # the library's instantiation follows the window set last: select it here (repet_istft itself only uses the
    # window's length and COLA gain)
    handle.set_window(window_function)
    half = window_length // 2
    number_channels, number_times, number_frequencies = spectrum.shape
    if number_frequencies != half + 1:
        raise ValueError("spectrum must hold window_length/2 + 1 bins")
    packed = np.empty((number_times, number_channels, half, 2), dtype=np.float32)
    packed[..., 0] = np.transpose(spectrum[:, :, :half].real, (1, 0, 2))
    packed[..., 1] = np.transpose(spectrum[:, :, :half].imag, (1, 0, 2))
    packed[:, :, 0, 1] = spectrum[:, :, half].real.T
    signal = np.empty((number_channels, (number_times - 1) * step_length), dtype=np.float32)
    gain = float(sum(window_function[0:window_length:step_length]))
    handle.check(handle.lib.repet_istft(handle.h, _ptr(packed), number_channels, number_times, gain, _ptr(signal)))
    return signal


def fast_stft_applies(window_length, step_length):
    return window_length in FAST_WINDOWS and 2 * step_length == window_length


def stft_general(audio_signal, window_function, step_length, handle=None):
    """_stft (repet.py:1001-1060) for ANY window length and step, float64 on the device: (S,) -> complex128
    (window_length, number_times), every bin, the reference's own layout."""
    handle = handle or get_handle()
    signal = np.ascontiguousarray(audio_signal, dtype=np.float64)
    window = np.ascontiguousarray(window_function, dtype=np.float64)
    if signal.ndim != 1 or window.ndim != 1:
        raise ValueError("audio_signal and window_function must be one-dimensional")
    window_length, step_length = len(window), int(step_length)
    number_times = handle.lib.repet_stft_frames(len(signal), window_length, step_length)
    audio_stft = np.empty((window_length, max(number_times, 0)), dtype=np.complex128)
    frames = ctypes.c_int32(0)
    handle.check(handle.lib.repet_stft_f64(handle.h, _ptr(signal), len(signal), _ptr(window), window_length, step_length,
                                           _ptr(audio_stft), ctypes.byref(frames)))
    assert frames.value == number_times
    return audio_stft


def istft_general(audio_stft, window_function, step_length, handle=None):
    """_istft (repet.py:1063-1105) for ANY window length and step, float64 on the device: complex (window_length,
    number_times) -> float64 (number_times * step - (window_length - step),)."""
    handle = handle or get_handle()
    spectrum = np.ascontiguousarray(audio_stft, dtype=np.complex128)
    window = np.ascontiguousarray(window_function, dtype=np.float64)
    window_length, number_times = spectrum.shape
    if len(window) != window_length:
        raise ValueError("operands could not be broadcast together (window length differs from the STFT's)")
    step_length = int(step_length)
    number_samples = max(0, number_times * step_length - (window_length - step_length))
    signal = np.empty(number_samples, dtype=np.float64)
    produced = _c_i64(0)
    handle.check(handle.lib.repet_istft_f64(handle.h, _ptr(spectrum), window_length, number_times, _ptr(window), step_length,
                                            _ptr(signal), ctypes.byref(produced)))
    assert produced.value == number_samples
    return signal


def acorr_general(data_matrix, handle=None):
    """_acorr (repet.py:1108-1139) for any number of rows, float64 on the device."""
    handle = handle or get_handle()
    data = np.ascontiguousarray(data_matrix, dtype=np.float64)
    rows, columns = data.shape
    out = np.empty((rows, columns), dtype=np.float64)
    handle.check(handle.lib.repet_acorr_f64(handle.h, _ptr(data), rows, columns, _ptr(out)))
    return out


def beatspectrum_general(audio_spectrogram, handle=None):
    """_beatspectrum (repet.py:1142-1158) for any size, float64 on the device: (F, T) -> (T,)."""
    handle = handle or get_handle()
    spectrogram = np.ascontiguousarray(audio_spectrogram, dtype=np.float64)
    number_frequencies, number_times = spectrogram.shape
    beat = np.empty(number_times, dtype=np.float64)
    handle.check(handle.lib.repet_beatspectrum_f64(handle.h, _ptr(spectrogram), number_frequencies, number_times, _ptr(beat)))
    return beat


def beatspectrum(audio_spectrogram, handle=None):
    """_beatspectrum (repet.py:1142-1158): (F, T) magnitudes -> float64 (T,).  Spectrograms that fit the drivers'
    fp32 beat kernel (T <= 1024 frames, F <= 1025) go through it; anything larger takes the float64 general path."""
    handle = handle or get_handle()
    if np.shape(audio_spectrogram)[1] > 1024 or np.shape(audio_spectrogram)[0] > 1025:
        return beatspectrum_general(audio_spectrogram, handle=handle)
    spectrogram = np.ascontiguousarray(np.asarray(audio_spectrogram).T, dtype=np.float32)  # time major
    number_times, number_rows = spectrogram.shape
    beat = np.empty(number_times, dtype=np.float64)
    handle.check(handle.lib.repet_beatspectrum(handle.h, _ptr(spectrogram), number_times, number_rows, _ptr(beat)))
    return beat


def period_of(audio_spectrogram, period_range2, handle=None):
    """_periods(_beatspectrum(V), period_range2) (repet.py:1249-1291) for one spectrogram."""
    handle = handle or get_handle()
    spectrogram = np.ascontiguousarray(np.asarray(audio_spectrogram).T, dtype=np.float32)
    number_times, number_rows = spectrogram.shape
    period = np.zeros(1, dtype=np.int32)
    handle.check(
        handle.lib.repet_period(
            handle.h, _ptr(spectrogram), number_times, number_rows, int(period_range2[0]), int(period_range2[1]), _ptr(period)
        )
    )
    return int(period[0])


def _select_bins(handle, number_frequencies):
    """The mask helpers take whole magnitude spectrograms: F = window_length/2 + 1 selects the
    library instantiation (the window set last decides, include/repet_b200.h)."""
    if number_frequencies not in (257, 513, 1025):
        raise NotImplementedError("spectrograms of 257, 513 or 1025 bins (window_length 512, 1024, 2048) are supported")
    handle.ensure_window(2 * (number_frequencies - 1))


def mask(audio_spectrogram, repeating_period, handle=None):
    """_mask (repet.py:1386-1458): (F, T) magnitudes, period -> float64 (F, T)."""
    handle = handle or get_handle()
    magnitude = np.ascontiguousarray(np.asarray(audio_spectrogram).T, dtype=np.float32)
    number_times, number_frequencies = magnitude.shape
    _select_bins(handle, number_frequencies)
    out = np.empty((number_times, number_frequencies), dtype=np.float32)
    handle.check(handle.lib.repet_mask(handle.h, _ptr(magnitude), number_times, int(repeating_period), _ptr(out)))
    return out.T.astype(np.float64)


def separate_f64(method, audio_signal, sampling_frequency, tunables, handle=None, spectrograms=True):
    """One call for the reference's documented usage (README.md:64-81): background by `method`,
    foreground = audio - background, and the display spectrograms abs(_stft(mean(x, axis=1)))[0:F] of
    mixture, background and foreground, all produced on the device from the buffers already there.
    Returns a dict: background, foreground (number_samples, number_channels) float64;
    audio_spectrogram, background_spectrogram, foreground_spectrogram (number_frequencies, number_times)
    float64 (when `spectrograms`); integers = the method's integer output (period(s) or packed lists)."""
    if method not in METHODS:
        raise ValueError("method must be one of %s" % sorted(METHODS))
    params, window_function = derive_params(sampling_frequency, tunables, method)
    return _run_f64(method, audio_signal, params, window_function, handle, foreground=True, spectrograms=spectrograms)


def spectrogram_batch_device(audio_ptr, spectrogram_ptr, number_clips, number_channels, number_samples,
                             sampling_frequency, tunables, handle=None):
    """Display spectrograms |STFT(mean_c x)| of device-resident fp32 planar clips (raw device pointers):
    spectrogram (clips, frames, pitch) fp32 with pitch = repet_spectrogram_pitch.  Returns (frames, pitch)."""
    handle = handle or get_handle()
    params, _ = derive_params(sampling_frequency, tunables)
    handle.ensure_window(params.window_length)
    handle.check(
        handle.lib.repet_spectrogram_batch_dev(
            handle.h, _vp(audio_ptr), number_clips, number_channels, number_samples, ctypes.byref(params),
            _vp(spectrogram_ptr),
        )
    )
    return (handle.lib.repet_spectrogram_frames(ctypes.byref(params), number_samples),
            handle.lib.repet_spectrogram_pitch(ctypes.byref(params)))


def foreground_device(audio_ptr, background_ptr, foreground_ptr, number_elements, handle=None):
    """foreground = audio - background over device-resident fp32 buffers (raw device pointers)."""
    handle = handle or get_handle()
    handle.check(handle.lib.repet_foreground_dev(handle.h, _vp(audio_ptr), _vp(background_ptr), number_elements,
                                                 _vp(foreground_ptr)))


def extended_f64(audio_signal, sampling_frequency, tunables, handle=None, return_periods=False):
    """repet.extended with the reference's calling convention (repet.py:205-419)."""
    params, window_function = derive_params(sampling_frequency, tunables, "extended")
    result = _run_f64("extended", audio_signal, params, window_function, handle)
    return (result["background"], result["integers"]) if return_periods else result["background"]


def adaptive_f64(audio_signal, sampling_frequency, tunables, handle=None, return_periods=False):
    """repet.adaptive with the reference's calling convention (repet.py:422-568)."""
    params, window_function = derive_params(sampling_frequency, tunables, "adaptive")
    result = _run_f64("adaptive", audio_signal, params, window_function, handle)
    return (result["background"], result["integers"]) if return_periods else result["background"]


def driver_batch(driver, audio, sampling_frequency, tunables, handle=None):
    """original / extended / adaptive over a batch: audio (B, C, S) float32 planar host memory.
    Returns (background (B, C, S) float32, integer outputs (B, ints_per_clip) int32)."""
    if driver not in METHODS:
        raise ValueError("unknown driver %r" % driver)
    params, window_function = derive_params(sampling_frequency, tunables, driver)
    return _run_batch(driver, audio, params, window_function, handle)


class PinnedArray:
    """A NumPy array on page-locked host memory (repet_host_alloc): host-buffer batch calls copy from / into it at
    the full rate of the host link, pageable arrays are staged by the driver at a fraction of it.  `.array` is
    the ndarray; the memory is released when the object is (keep it alive while views of the array are in use)."""

    def __init__(self, shape, dtype):
        self.lib = load_library()
        dtype = np.dtype(dtype)
        number_bytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
        pointer = _vp()
        rc = self.lib.repet_host_alloc(ctypes.byref(pointer), max(1, number_bytes))
        if rc != REPET_OK:
            raise MemoryError("repet_host_alloc(%d bytes) failed with status %d" % (number_bytes, rc))
        self.pointer = pointer
        buffer = (ctypes.c_char * max(1, number_bytes)).from_address(pointer.value)
        self.array = np.frombuffer(buffer, dtype=dtype, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)

    def close(self):
        if getattr(self, "pointer", None):
            self.array = None
            self.lib.repet_host_free(self.pointer)
            self.pointer = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def device_count():
    return int(load_library().repet_device_count())


def shard_bounds(number_clips, number_shards):
    """Contiguous balanced split of `number_clips` over `number_shards`: list of (first, stop).  The same split as
    repet_shard.shard_range (one process per GPU); here one host thread per GPU."""
    base, extra = divmod(int(number_clips), int(number_shards))
    bounds, first = [], 0
    for r in range(int(number_shards)):
        stop = first + base + (1 if r < extra else 0)
        bounds.append((first, stop))
        first = stop
    return bounds


def separate_batch(driver, audio, sampling_frequency, tunables, handle=None, in_format="f32", out_format="f32",
                   out=None, devices=None):
    """Any driver over a batch of equally long clips in host memory (repet_separate_batch).

    audio: (B, C, S) float32 planar (`in_format="f32"`) or (B, S, C) int16 PCM in WAV order (`"pcm16"`: what
    scipy.io.wavfile.read returns, normalised by 2^15 on the device as repet.wavread does, repet.py:929).
    Output: background in `out_format` -- "f32" (B, C, S) float32, or "pcm16" (B, S, C) int16 = round(y * 2^15)
    saturated (lossy) -- and the integer outputs (B, ints_per_clip) int32.

    `devices`: a sequence of GPU indices shards the batch by clip over them inside this process, one handle and
    one host thread per GPU over the same C entry point (clips are independent: no collective, SURVEY.md 8(e))."""
    if driver not in METHODS:
        raise ValueError("unknown driver %r" % driver)
    params, window_function = derive_params(sampling_frequency, tunables, driver)
    return _run_batch(driver, audio, params, window_function, handle, in_format, out_format, out, devices)


# ------------------------------------------------------------------------------------------
# one long track over several GPUs, by time block (SURVEY.md 8(e), "finer partitions")
# ------------------------------------------------------------------------------------------
def _run_shards(jobs, devices):
    """jobs: list of callables f(handle) -> result, shard k runs on devices[k % len(devices)]; one host thread per
    DISTINCT device (a handle is not re-entrant), shards of a device in order.  Returns the results in job order."""
    devices = [int(d) for d in devices]
    if not devices:
        raise ValueError("devices must name at least one GPU")
    results = [None] * len(jobs)
    errors = []
    by_device = {}
    for k in range(len(jobs)):
        by_device.setdefault(devices[k % len(devices)], []).append(k)
    handles = {d: get_handle(d) for d in by_device}

    def worker(device):
        try:
            for k in by_device[device]:
                results[k] = jobs[k](handles[device])
        except BaseException as exc:  # re-raised on the caller's thread
            errors.append(exc)

    threads = [threading.Thread(target=worker, args=(d,)) for d in by_device]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return results


def track_time_blocks(driver, number_samples, params, number_shards):
    """Sample ranges [a, b) that split ONE track of `driver` into `number_shards` time blocks whose separate
    separations can be merged into exactly the whole-track result (pure host logic, tested on CPU):

    extended   cuts at multiples of the segment step: block k holds whole 10 s segments, the last segment of a block
               has the regular length (only the track's last segment absorbs the remainder, repet.py:320-322)
    adaptive   cuts at multiples of the beat-spectrogram step in samples: the segment grid (repet.py:1194) is anchored
               at frame 0 of every block exactly as in the whole track
    simonline  cuts at multiples of the hop: every block replays its similarity history (buffer_frames - 1 frames)
               through online_frame_base
    Returns a list of (a, b); fewer than number_shards entries when the track is too short to cut."""
    S, K = int(number_samples), max(1, int(number_shards))
    if driver == "extended":
        seg_len, step = params.segment_length, params.segment_step
        if S < seg_len + step:
            return [(0, S)]
        n_seg = 1 + (S - seg_len) // step
        K = min(K, n_seg)
        cuts = [0]
        for k in range(1, K):
            m = (n_seg * k) // K  # first segment of block k
            if m * step > cuts[-1]:
                cuts.append(m * step)
        return [(a, b) for a, b in zip(cuts, cuts[1:] + [S])]
    if driver == "adaptive":
        unit = params.segment_step * params.step_length
    elif driver == "simonline":
        unit = params.step_length
    else:
        raise ValueError("time-block sharding applies to extended, adaptive and simonline")
    n_units = S // unit
    K = min(K, max(1, n_units))
    if driver == "simonline":
        # the first block must get through the reference's warm-up on its own (repet.py:794-810)
        K = min(K, max(1, S // ((params.buffer_frames + 1) * unit)))
    cuts = sorted({(n_units * k) // K * unit for k in range(K)})
    return [(a, b) for a, b in zip(cuts, cuts[1:] + [S])]


def sharded_track(driver, audio_signal, sampling_frequency, tunables, devices):
    """ONE long track split by time block over several GPUs (one handle and one host thread per GPU; more blocks
    than GPUs run in turn).  The merged output equals the single-call result: to rounding for `extended` (the
    junction cross-fade is applied in float64 on the host, repet.py:398-409) and `adaptive` (every block is
    separated with a halo that covers the beat-spectrogram segments and the median taps of its frames, and only
    its own samples are kept), bit for bit for `simonline` (each block replays its similarity history)."""
    x = np.ascontiguousarray(audio_signal, dtype=np.float64)
    number_samples, _ = x.shape
    params, window_function = derive_params(sampling_frequency, tunables, driver)
    blocks = track_time_blocks(driver, number_samples, params, len(list(devices)))
    if len(blocks) == 1:
        return {"extended": extended_f64, "adaptive": adaptive_f64, "simonline": simonline_f64}[driver](
            x, sampling_frequency, tunables)
    out = np.empty_like(x)
    if driver == "extended":
        seg_len, step = params.segment_length, params.segment_step
        overlap = seg_len - step
        # block k = samples [a_k, b_k + overlap): its last segment reaches `overlap` samples into the next block
        jobs = [(lambda h, a=a, b=b: extended_f64(x[a : min(b + overlap, number_samples)], sampling_frequency, tunables,
                                                  handle=h)) for a, b in blocks]
        parts = _run_shards(jobs, devices)
        import scipy.signal.windows

        window = scipy.signal.windows.triang(2 * overlap)  # repet.py:284
        for (a, b), y in zip(blocks, parts):
            if a == 0:
                out[: len(y)] = y
            else:
                # the reference's in-place step for the block's first segment (repet.py:398-409): what is already
                # there fades out, the new segment fades in, the rest is the block's own
                out[a : a + overlap] = out[a : a + overlap] * window[overlap:, None] + y[:overlap] * window[:overlap, None]
                out[a + overlap : a + len(y)] = y[overlap:]
        return out
    if driver == "adaptive":
        unit = params.segment_step * params.step_length
        halo = 3 * unit  # beat segments reach 1 step, the 5 median taps 2 periods (< 2 steps) beyond a frame
        jobs = []
        for a, b in blocks:
            lo, hi = max(0, a - halo), min(number_samples, b + halo)
            jobs.append(lambda h, lo=lo, hi=hi, a=a, b=b: adaptive_f64(x[lo:hi], sampling_frequency, tunables, handle=h)[a - lo : b - lo])
        for (a, b), y in zip(blocks, _run_shards(jobs, devices)):
            out[a:b] = y
        return out
    # simonline: a block is a window of the stream -- its samples plus the history its first frames look back on
    N, H, B = params.window_length, params.step_length, params.buffer_frames
    if (B - 2) * H + N > number_samples:
        raise ValueError("operands could not be broadcast together (signal shorter than the buffer)")

    def online_block(h, a, b):
        first_block = a // H
        first_needed = max(0, first_block - 1)  # output hop b mixes frames b - 1 and b
        first_frame = max(0, first_needed - (B - 1))
        lo = first_frame * H
        # frames that touch [a, b): up to the one starting below b; the window must hold whole frames
        last_frame = min((b - 1) // H, max(0, -(-(number_samples - N) // H)))
        hi = min(number_samples, last_frame * H + N)
        p = RepetParams.from_buffer_copy(params)
        p.online_frame_base = int(first_frame)
        return _run_f64("simonline", x[lo:hi], p, window_function, h)["background"][a - lo : b - lo]

    jobs = [(lambda h, a=a, b=b: online_block(h, a, b)) for a, b in blocks]
    for (a, b), y in zip(blocks, _run_shards(jobs, devices)):
        out[a:b] = y
    return out


def ragged_groups(shapes):
    """Group clip indices by (channels, samples): clips of equal shape go through one batch call.  Pure host
    logic (the groups are returned in order of first appearance, indices ascending inside a group)."""
    groups = {}
    for index, shape in enumerate(shapes):
        if len(shape) != 2:
            raise ValueError("every clip must have shape (channels, samples)")
        groups.setdefault((int(shape[0]), int(shape[1])), []).append(index)
    return list(groups.items())


def driver_batch_ragged(driver, clips, sampling_frequency, tunables, handle=None):
    """A batch of clips of DIFFERENT lengths (a list of (C, S_i) float32 arrays): clips are never padded
    -- a clip's frame count, period range and periods depend on its length (repet.py:165-173) -- but grouped
    by shape, one batch call per group.  Returns (list of backgrounds, list of integer outputs) in input order."""
    clips = [np.asarray(c, dtype=np.float32) for c in clips]
    backgrounds = [None] * len(clips)
    integers = [None] * len(clips)
    for (channels, samples), members in ragged_groups([c.shape for c in clips]):
        stacked = np.stack([clips[i] for i in members]) if members else np.zeros((0, channels, samples), np.float32)
        if driver == "original":
            background, ints = original_batch(stacked, sampling_frequency, tunables, handle=handle)
            ints = ints[:, None]
        else:
            background, ints = driver_batch(driver, stacked, sampling_frequency, tunables, handle=handle)
        for slot, index in enumerate(members):
            backgrounds[index] = background[slot]
            integers[index] = ints[slot]
    return backgrounds, integers


def beatspectrogram(audio_spectrogram, segment_length, segment_step, handle=None):
    """_beatspectrogram (repet.py:1161-1206): (F, T) -> float64 (segment_length, T).  The device
    computes the beat spectrum of every segment; the column replication (including the all-zero
    column i+step-1, quirk Q3) is pure data movement and happens here."""
    handle = handle or get_handle()
    spectrogram = np.ascontiguousarray(np.asarray(audio_spectrogram).T, dtype=np.float32)
    number_times, number_rows = spectrogram.shape
    number_segments = -(-number_times // segment_step)
    beat = np.empty((number_segments, segment_length), dtype=np.float64)
    count = ctypes.c_int32(0)
    handle.check(
        handle.lib.repet_beatspectrogram(
            handle.h, _ptr(spectrogram), number_times, number_rows, int(segment_length), int(segment_step), _ptr(beat),
            ctypes.byref(count),
        )
    )
    assert count.value == number_segments
    beat_spectrogram = np.zeros((segment_length, number_times))
    for index, i in enumerate(range(0, number_times, segment_step)):
        beat_spectrogram[:, i] = beat[index]
        beat_spectrogram[:, i : min(i + segment_step - 1, number_times)] = beat[index][:, np.newaxis]
    return beat_spectrogram


def periods(beat_spectrogram, period_range, handle=None):
    """_periods (repet.py:1249-1291): 1-D beat spectrum -> int, 2-D beat spectrogram -> int array."""
    handle = handle or get_handle()
    beat = np.ascontiguousarray(beat_spectrogram, dtype=np.float64)
    one_dimensional = beat.ndim == 1
    matrix = beat.reshape(beat.shape[0], -1)
    out = np.zeros(matrix.shape[1], dtype=np.int32)
    handle.check(
        handle.lib.repet_periods(
            handle.h, _ptr(matrix), matrix.shape[0], matrix.shape[1], int(period_range[0]), int(period_range[1]), _ptr(out)
        )
    )
    return int(out[0]) if one_dimensional else out.astype(np.int64)


def adaptivemask(audio_spectrogram, repeating_periods, filter_order, handle=None):
    """_adaptivemask (repet.py:1461-1508): (F, T) magnitudes, per-frame periods -> float64 (F, T)."""
    handle = handle or get_handle()
    magnitude = np.ascontiguousarray(np.asarray(audio_spectrogram).T, dtype=np.float32)
    number_times, number_frequencies = magnitude.shape
    _select_bins(handle, number_frequencies)
    per = np.ascontiguousarray(repeating_periods, dtype=np.int32)
    if per.shape != (number_times,):
        raise ValueError("one period per time frame expected")
    out = np.empty((number_times, number_frequencies), dtype=np.float32)
    handle.check(handle.lib.repet_adaptivemask(handle.h, _ptr(magnitude), number_times, _ptr(per), int(filter_order), _ptr(out)))
    return out.T.astype(np.float64)


def unpack_lists(ints, number_frames, number):
    """[counts T][indices T x number] (the ABI's per-clip layout) -> list of T int arrays."""
    counts = ints[:number_frames]
    table = ints[number_frames : number_frames * (number + 1)].reshape(number_frames, number)
    return [table[i, : counts[i]].astype(np.int64) for i in range(number_frames)]


def sim_f64(audio_signal, sampling_frequency, tunables, handle=None, return_indices=False):
    """repet.sim with the reference's calling convention (repet.py:571-709)."""
    params, window_function = derive_params(sampling_frequency, tunables, "sim")
    result = _run_f64("sim", audio_signal, params, window_function, handle)
    if return_indices:
        ints, number = result["integers"], params.similarity_number
        return result["background"], unpack_lists(ints, len(ints) // (number + 1), number)
    return result["background"]


def simonline_f64(audio_signal, sampling_frequency, tunables, handle=None, return_indices=False):
    """repet.simonline with the reference's calling convention (repet.py:712-911).  With
    return_indices the lists of frames >= buffer_frames-1 hold FRAME indices (most similar first)."""
    params, window_function = derive_params(sampling_frequency, tunables, "simonline")
    result = _run_f64("simonline", audio_signal, params, window_function, handle)
    if return_indices:
        ints, number = result["integers"], params.similarity_number
        return result["background"], unpack_lists(ints, len(ints) // (number + 1), number)
    return result["background"]


def selfsimilarity(data_matrix, handle=None):
    """_selfsimilaritymatrix (repet.py:1209-1225), the device's fast pass: (F, T) -> float32 (T, T)."""
    handle = handle or get_handle()
    magnitude = np.ascontiguousarray(np.asarray(data_matrix).T, dtype=np.float32)
    number_times, number_rows = magnitude.shape
    out = np.empty((number_times, number_times), dtype=np.float32)
    handle.check(handle.lib.repet_selfsimilarity(handle.h, _ptr(magnitude), number_times, number_rows, _ptr(out)))
    return out


def similaritymatrix(data_matrix1, data_matrix2, handle=None):
    """_similaritymatrix (repet.py:1228-1246) in exact float64: (F, T1), (F, T2) -> (T1, T2)."""
    handle = handle or get_handle()
    m1 = np.ascontiguousarray(np.asarray(data_matrix1).T, dtype=np.float32)
    m2 = np.ascontiguousarray(np.asarray(data_matrix2).T, dtype=np.float32)
    if m1.shape[1] != m2.shape[1]:
        raise ValueError("matrices must have the same number of rows")
    out = np.empty((m1.shape[0], m2.shape[0]), dtype=np.float64)
    handle.check(handle.lib.repet_similarity(handle.h, _ptr(m1), m1.shape[0], _ptr(m2), m2.shape[0], m1.shape[1], _ptr(out)))
    return out


def localmaxima(data_vector, minimum_value, minimum_distance, number_values, handle=None):
    """_localmaxima (repet.py:1294-1345): values and indices of the strict local maxima, best first."""
    handle = handle or get_handle()
    data = np.ascontiguousarray(data_vector, dtype=np.float64).reshape(-1, 1)
    number = max(1, int(number_values))
    idx = np.zeros((1, number), dtype=np.int32)
    val = np.zeros((1, number), dtype=np.float64)
    cnt = np.zeros(1, dtype=np.int32)
    handle.check(handle.lib.repet_localmaxima(handle.h, _ptr(data), data.shape[0], 1, float(minimum_value),
                                              int(minimum_distance), number, _ptr(idx), _ptr(cnt), _ptr(val)))
    n = min(int(cnt[0]), int(number_values))
    return val[0, :n].copy(), idx[0, :n].astype(np.int64)


def indices(similarity_matrix, similarity_threshold, similarity_distance, similarity_number, handle=None):
    """_indices (repet.py:1348-1383): the local-maximum indices of every column, as a list of arrays."""
    handle = handle or get_handle()
    data = np.ascontiguousarray(similarity_matrix, dtype=np.float64)
    n, columns = data.shape
    number = max(1, int(similarity_number))
    idx = np.zeros((columns, number), dtype=np.int32)
    cnt = np.zeros(columns, dtype=np.int32)
    handle.check(handle.lib.repet_localmaxima(handle.h, _ptr(data), n, columns, float(similarity_threshold),
                                              int(similarity_distance), number, _ptr(idx), _ptr(cnt), None))
    return [idx[c, : min(int(cnt[c]), int(similarity_number))].astype(np.int64) for c in range(columns)]


def simmask(audio_spectrogram, similarity_indices, handle=None):
    """_simmask (repet.py:1511-1545): (F, T) magnitudes + list of index arrays -> float64 (F, T)."""
    handle = handle or get_handle()
    magnitude = np.ascontiguousarray(np.asarray(audio_spectrogram).T, dtype=np.float32)
    number_times, number_frequencies = magnitude.shape
    _select_bins(handle, number_frequencies)
    number = max(1, max((len(v) for v in similarity_indices), default=1))
    idx = np.zeros((number_times, number), dtype=np.int32)
    cnt = np.zeros(number_times, dtype=np.int32)
    for i, values in enumerate(similarity_indices):
        cnt[i] = len(values)
        idx[i, : len(values)] = values
    out = np.empty((number_times, number_frequencies), dtype=np.float32)
    handle.check(handle.lib.repet_simmask(handle.h, _ptr(magnitude), number_times, _ptr(idx), _ptr(cnt), number, _ptr(out)))
    return out.T.astype(np.float64)


def acorr(data_matrix, handle=None):
    """_acorr (repet.py:1108-1139): unbiased autocorrelation of every column, (rows, cols) -> float64."""
    handle = handle or get_handle()
    if 2 * np.shape(data_matrix)[0] - 1 > 2048:
        return acorr_general(data_matrix, handle=handle)  # more rows than the drivers' 2048-point transform holds
    data = np.ascontiguousarray(data_matrix, dtype=np.float32)
    rows, columns = data.shape
    out = np.empty((rows, columns), dtype=np.float64)
    handle.check(handle.lib.repet_acorr(handle.h, _ptr(data), rows, columns, _ptr(out)))
    return out


def original_batch_pcm16(pcm, sampling_frequency, tunables, handle=None):
    """`original` over int16 PCM clips in WAV order: pcm (B, S, C) int16 -> (background (B, C, S) float32,
    periods (B,) int32).  The samples are normalised by 2^15 on the device, as repet.wavread does."""
    params, window_function = derive_params(sampling_frequency, tunables)
    background, ints = _run_batch("original", pcm, params, window_function, handle, in_format="pcm16")
    return background, ints[:, 0]


class SimOnlineStreamHost:
    """Host-side reference implementation of the stream (kept for cross-checks; `SimOnlineStream` below is the
    product path): block-wise online REPET-SIM (repet.py:712-911) with the results of one whole-signal call.

    `process(block)` takes the next samples (n, channels) and returns the background samples that have
    become final (every frame covering them is complete: a latency of one hop, 1024 samples at 44.1 kHz);
    `flush()` returns the rest, zero-padding the last frame as the reference does.  Each call re-analyses
    the last buffer_length seconds on the device (the path runs at >70 000x realtime, so this costs a
    fraction of a millisecond per second of audio) with the ring-slot order of the whole stream
    (`online_frame_base`, quirk Q6).  Like the reference, nothing is synthesised before frame
    buffer_frames-1: the first ~10 s of output are zero.
    """

    def __init__(self, sampling_frequency, number_channels, tunables, handle=None):
        self.handle = handle or get_handle()
        self.fs = sampling_frequency
        self.channels = int(number_channels)
        self.tunables = dict(tunables)
        self.params, self.window_function = derive_params(sampling_frequency, self.tunables, "simonline")
        self.N, self.H, self.B = self.params.window_length, self.params.step_length, self.params.buffer_frames
        self.buffer = np.zeros((0, self.channels), dtype=np.float64)  # samples from frame `buffer_frame0` on
        self.buffer_frame0 = 0
        self.received = 0
        self.emitted = 0

    def _run_window(self, first_frame, number_samples):
        """simonline on buffer samples [first_frame*H - buffer_frame0*H, ... + number_samples)."""
        lo = (first_frame - self.buffer_frame0) * self.H
        params = RepetParams.from_buffer_copy(self.params)
        params.online_frame_base = int(first_frame)
        return _run_f64("simonline", self.buffer[lo : lo + number_samples], params, self.window_function,
                        self.handle)["background"]

    def _advance(self, final_until, total_samples_for_window):
        """Emit background samples [emitted, final_until)."""
        if final_until <= self.emitted:
            return np.zeros((0, self.channels))
        first_block = self.emitted // self.H
        first_needed = max(0, first_block - 1)  # block b mixes frames b-1 and b
        first_frame = max(0, first_needed - (self.B - 1))  # ... and their similarity history
        first_frame = max(first_frame, self.buffer_frame0)
        out = self._run_window(first_frame, total_samples_for_window - first_frame * self.H)
        lo = self.emitted - first_frame * self.H
        chunk = out[lo : lo + (final_until - self.emitted)]
        self.emitted = final_until
        # drop samples no later window will need
        keep_frame = max(0, self.emitted // self.H - 1 - (self.B - 1))
        if keep_frame > self.buffer_frame0:
            self.buffer = self.buffer[(keep_frame - self.buffer_frame0) * self.H :]
            self.buffer_frame0 = keep_frame
        return chunk

    def process(self, block):
        block = np.asarray(block, dtype=np.float64)
        if block.ndim != 2 or block.shape[1] != self.channels:
            raise ValueError("block must have shape (samples, %d)" % self.channels)
        self.buffer = np.concatenate((self.buffer, block), axis=0)
        self.received += block.shape[0]
        if self.received < self.N:
            return np.zeros((0, self.channels))
        last_complete = (self.received - self.N) // self.H
        final_until = (last_complete + 1) * self.H
        if last_complete < self.B - 1:
            # nothing is synthesised yet (quirk Q5): the final samples are zeros
            chunk = np.zeros((max(0, final_until - self.emitted), self.channels))
            self.emitted = max(self.emitted, final_until)
            return chunk
        return self._advance(final_until, last_complete * self.H + self.N)

    def flush(self):
        """End of stream: everything up to the last received sample."""
        if self.received <= self.emitted:
            return np.zeros((0, self.channels))
        if self.received < (self.B - 2) * self.H + self.N:
            raise ValueError("operands could not be broadcast together (signal shorter than the buffer)")
        return self._advance(self.received, self.received)


class SimOnlineStream:
    """Block-wise online REPET-SIM (repet.py:712-911) on the stateful C stream (repet_simonline_open / _block /
    _flush / _close): the last buffer_length seconds of samples live in device memory, a block costs one upload of
    the new samples and one download of the samples that became final.

    `process(block)` takes the next samples (n, channels) and returns the background samples that have become
    final (every frame covering them is complete: a latency of one hop, 1024 samples at 44.1 kHz); `flush()`
    returns the rest, zero-padding the last frame as the reference does.  The concatenated outputs equal
    `repet.simonline` on the whole signal (ring-slot order of the whole stream, quirk Q6); like the reference,
    nothing is synthesised before frame buffer_frames-1: the first ~10 s of output are zero."""

    def __init__(self, sampling_frequency, number_channels, tunables, handle=None):
        self.handle = handle or get_handle()
        self.channels = int(number_channels)
        self.params, _ = derive_params(sampling_frequency, dict(tunables), "simonline")
        self.handle.ensure_window(self.params.window_length)
        self._stream = _vp()
        self.handle.check(self.handle.lib.repet_simonline_open(self.handle.h, ctypes.byref(self.params), self.channels,
                                                               ctypes.byref(self._stream)))

    def _call(self, fn, block):
        hop = self.params.step_length
        capacity = (0 if block is None else block.shape[0]) + 2 * hop if fn == "block" else self._pending + 2 * hop
        out = np.empty((capacity, self.channels), dtype=np.float64)
        n_out = _c_i64(0)
        lib = self.handle.lib
        if fn == "block":
            rc = lib.repet_simonline_block(self._stream, _ptr(block), block.shape[0], _ptr(out), capacity, ctypes.byref(n_out))
        else:
            rc = lib.repet_simonline_flush(self._stream, _ptr(out), capacity, ctypes.byref(n_out))
        self.handle.check(rc)
        return out[: n_out.value]

    _pending = 0  # samples received and not yet emitted (bounds the flush buffer)

    def process(self, block):
        block = np.ascontiguousarray(block, dtype=np.float64)
        if block.ndim != 2 or block.shape[1] != self.channels:
            raise ValueError("block must have shape (samples, %d)" % self.channels)
        self.handle.ensure_window(self.params.window_length)
        out = self._call("block", block)
        self._pending += block.shape[0] - out.shape[0]
        return out

    def flush(self):
        """End of stream: everything up to the last received sample."""
        self.handle.ensure_window(self.params.window_length)
        out = self._call("flush", None)
        self._pending -= out.shape[0]
        return out

    def close(self):
        if self._stream:
            self.handle.lib.repet_simonline_close(self._stream)
            self._stream = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
