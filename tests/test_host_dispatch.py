"""CPU: the binding's choice between the fast kernels and the general float64 path, on a fake library.

Every separation call runs on the fast kernels (repet_separate_f64 / repet_separate_batch, after the window upload)
unless the input is a shape they are not compiled for (96 kHz, more than two channels) or they refuse it
(REPET_E_UNSUPPORTED); then it runs on repet_general_f64, clip by clip for a batch.  No other error is retried.
The fake records every call and answers each entry point with the status a test sets."""

import ctypes
import itertools

import numpy as np
import pytest

import repet
from repet import _host

FAST_F64, FAST_BATCH, GENERAL = "repet_separate_f64", "repet_separate_batch", "repet_general_f64"
ENTRY_POINTS = ("repet_set_window", FAST_F64, FAST_BATCH, GENERAL, "repet_stft_f64")


class FakeLibrary:
    """The symbols the separation calls use.  `refuse[name] = n`: the next n calls answer REPET_E_UNSUPPORTED;
    `fail[name] = status`: every call answers `status`."""

    def __init__(self):
        self.calls = []
        self.refuse = {}
        self.fail = {}
        self._handles = itertools.count(1)

    def _answer(self, name, *args):
        self.calls.append((name, args))
        if self.refuse.get(name, 0) > 0:
            self.refuse[name] -= 1
            return _host.REPET_E_UNSUPPORTED
        return self.fail.get(name, _host.REPET_OK)

    def count(self, name):
        return sum(1 for call, _ in self.calls if call == name)

    def repet_create(self, device, out):
        out._obj.value = next(self._handles)
        return _host.REPET_OK

    def repet_destroy(self, h):
        return _host.REPET_OK

    def repet_last_error(self, h):
        return b"fake"

    def repet_set_window(self, h, window, n):
        self.calls.append(("repet_set_window", (h, window, n)))
        return _host.REPET_OK if n in _host.FAST_WINDOWS else _host.REPET_E_UNSUPPORTED

    def repet_ints_per_clip(self, method, p, n):  # repet_abi.cu
        p = p._obj
        T = (n + p.step_length - 1) // p.step_length + 1
        if method == 1:
            return 1 if n < p.segment_length + p.segment_step else 1 + (n - p.segment_length) // p.segment_step
        frames = 0 if n < p.window_length else (n - p.window_length + p.step_length - 1) // p.step_length + 1
        return {0: 1, 2: T, 3: T * (p.similarity_number + 1), 4: frames * (p.similarity_number + 1)}[method]

    def repet_spectrogram_frames(self, p, n):
        return (n + p._obj.step_length - 1) // p._obj.step_length + 1

    def repet_spectrogram_pitch(self, p):
        return (p._obj.window_length // 2 + 1 + 7) // 8 * 8

    def repet_stft_frames(self, n, window_length, step_length):
        return -(-(n + 2 * (window_length // 2) - window_length) // step_length) + 1

    def repet_stft_f64(self, h, signal, n, window, window_length, step_length, out, frames):
        frames._obj.value = self.repet_stft_frames(n, window_length, step_length)
        return self._answer("repet_stft_f64", h)

    def repet_separate_f64(self, h, method, audio, S, C, p, background, foreground, spectrograms, ints, capacity):
        ctypes.memset(background, 0, S * C * 8)
        return self._answer(FAST_F64, h, method, audio, S, C, p._obj.window_length, background, foreground,
                            spectrograms, ints, capacity)

    def repet_separate_batch(self, h, method, audio, in_format, n_clips, C, S, p, background, out_format, ints):
        ctypes.memset(background, 0, n_clips * C * S * (2 if out_format else 4))
        return self._answer(FAST_BATCH, h, method, audio, in_format, n_clips, C, S, p._obj.window_length,
                            background, out_format, ints)

    def repet_general_f64(self, h, method, audio, S, C, p, window, background, ints, capacity):
        ctypes.memset(background, 0, S * C * 8)
        return self._answer(GENERAL, h, method, audio, S, C, p._obj.window_length, window, background, ints, capacity)


@pytest.fixture
def fake(monkeypatch):
    library = FakeLibrary()
    monkeypatch.setattr(_host, "_lib", library)
    monkeypatch.setattr(_host, "_handles", {})
    return library


TUN = repet._tunables()
SECONDS = 24  # long enough for three `extended` segments and two `simonline` time blocks


def _derived(fs):
    params, _ = _host.derive_params(fs, TUN)
    return params.window_length, params.step_length


def _frames(fs):
    N, H = _derived(fs)
    return _host.number_of_frames(SECONDS * fs, N, H)


def _online_frames(fs):
    N, H = _derived(fs)
    return int(np.ceil((SECONDS * fs - N) / H)) + 1  # repet.py:781


def _clip(fs, channels):
    return np.zeros((SECONDS * fs, channels))


def _batch(fs, channels, clips=3):
    return np.zeros((clips, channels, SECONDS * fs), dtype=np.float32)


def _pcm(fs, channels, clips=3):
    return np.zeros((clips, SECONDS * fs, channels), dtype=np.int16)


def _signal(y, fs, channels):
    assert y.shape == (SECONDS * fs, channels) and y.dtype == np.float64


def _planar(y, fs, channels, clips=3, dtype=np.float32):
    assert y.shape == (clips, channels, SECONDS * fs) and y.dtype == dtype


def _integers(ints, shape):
    assert ints.shape == shape and ints.dtype == np.int32


def check_original(out, fs, C):
    y, period = out
    _signal(y, fs, C)
    assert isinstance(period, int)


def check_extended(out, fs, C):
    y, periods = out
    _signal(y, fs, C)
    _integers(periods, (1 + (SECONDS - TUN["segment_length"]) // TUN["segment_step"],))


def check_adaptive(out, fs, C):
    y, periods = out
    _signal(y, fs, C)
    _integers(periods, (_frames(fs),))


def check_sim(out, fs, C):
    y, lists = out
    _signal(y, fs, C)
    assert len(lists) == _frames(fs)


def check_simonline(out, fs, C):
    y, lists = out
    _signal(y, fs, C)
    assert len(lists) == _online_frames(fs)


def check_separate(out, fs, C):
    assert list(out) == ["background", "foreground", "integers", "audio_spectrogram", "background_spectrogram",
                         "foreground_spectrogram"]
    _signal(out["background"], fs, C)
    _signal(out["foreground"], fs, C)
    _integers(out["integers"], (_frames(fs),))
    N, _ = _derived(fs)
    for name in _host.SPECTROGRAMS:
        assert out[name].shape == (N // 2 + 1, _frames(fs)) and out[name].dtype == np.float64


def check_original_batch(out, fs, C):
    _planar(out[0], fs, C)
    _integers(out[1], (3,))


def check_driver_batch(out, fs, C):
    _planar(out[0], fs, C)
    _integers(out[1], (3, _frames(fs)))


def check_separate_batch_pcm16(out, fs, C):
    assert out[0].shape == (3, SECONDS * fs, C) and out[0].dtype == np.int16
    _integers(out[1], (3, _frames(fs) * (TUN["similarity_number"] + 1)))


def check_sharded_batch(out, fs, C):
    _planar(out[0], fs, C)
    _integers(out[1], (3, 1))


def check_track(out, fs, C):
    _signal(out, fs, C)


def run_stream_host(fs, C):
    x = _clip(fs, C)
    stream = _host.SimOnlineStreamHost(fs, C, TUN)
    return np.concatenate([stream.process(x), stream.flush()])


# name -> (call(fs, channels), fast entry point, fast calls, general calls, check)
CASES = {
    "original_f64": (lambda fs, C: _host.original_f64(_clip(fs, C), fs, TUN, return_period=True),
                     FAST_F64, 1, 1, check_original),
    "extended_f64": (lambda fs, C: _host.extended_f64(_clip(fs, C), fs, TUN, return_periods=True),
                     FAST_F64, 1, 1, check_extended),
    "adaptive_f64": (lambda fs, C: _host.adaptive_f64(_clip(fs, C), fs, TUN, return_periods=True),
                     FAST_F64, 1, 1, check_adaptive),
    "sim_f64": (lambda fs, C: _host.sim_f64(_clip(fs, C), fs, TUN, return_indices=True), FAST_F64, 1, 1, check_sim),
    "simonline_f64": (lambda fs, C: _host.simonline_f64(_clip(fs, C), fs, TUN, return_indices=True),
                      FAST_F64, 1, 1, check_simonline),
    "separate_f64": (lambda fs, C: _host.separate_f64("adaptive", _clip(fs, C), fs, TUN),
                     FAST_F64, 1, 1, check_separate),
    "original_batch": (lambda fs, C: _host.original_batch(_batch(fs, C), fs, TUN),
                       FAST_BATCH, 1, 3, check_original_batch),
    "original_batch_pcm16": (lambda fs, C: _host.original_batch_pcm16(_pcm(fs, C), fs, TUN),
                             FAST_BATCH, 1, 3, check_original_batch),
    "driver_batch": (lambda fs, C: _host.driver_batch("adaptive", _batch(fs, C), fs, TUN),
                     FAST_BATCH, 1, 3, check_driver_batch),
    "separate_batch": (lambda fs, C: _host.separate_batch("sim", _pcm(fs, C), fs, TUN, in_format="pcm16",
                                                          out_format="pcm16"),
                       FAST_BATCH, 1, 3, check_separate_batch_pcm16),
    "separate_batch_devices": (lambda fs, C: _host.separate_batch("original", _batch(fs, C), fs, TUN, devices=[0, 1]),
                               FAST_BATCH, 2, 3, check_sharded_batch),
    "sharded_track": (lambda fs, C: _host.sharded_track("simonline", _clip(fs, C), fs, TUN, devices=[0, 1]),
                      FAST_F64, 2, 2, check_track),
    "stream_host": (run_stream_host, FAST_F64, 2, 2, check_track),
}

FAST_SHAPE = (44100, 2)
GENERAL_SHAPES = [(96000, 2), (44100, 3)]


def _windows_precede_fast_calls(fake):
    """Every fast call comes after its handle's upload of the window it uses."""
    uploaded = set()
    for name, args in fake.calls:
        if name == "repet_set_window":
            uploaded.add((args[0].value, args[2]))
        elif name in (FAST_F64, FAST_BATCH):
            window_length = args[7] if name == FAST_BATCH else args[5]
            assert (args[0].value, window_length) in uploaded, "%s before its window" % name
    return True


@pytest.mark.parametrize("case", CASES)
def test_fast_shape_runs_the_fast_kernels_only(fake, case):
    call, entry, n_fast, _, check = CASES[case]
    check(call(*FAST_SHAPE), *FAST_SHAPE)
    assert fake.count(entry) == n_fast and fake.count(GENERAL) == 0
    assert fake.count(FAST_F64) + fake.count(FAST_BATCH) == n_fast
    assert _windows_precede_fast_calls(fake)


@pytest.mark.parametrize("shape", GENERAL_SHAPES, ids=["96kHz", "3ch"])
@pytest.mark.parametrize("case", CASES)
def test_general_shape_runs_the_general_path_only(fake, case, shape):
    call, _, _, n_general, check = CASES[case]
    check(call(*shape), *shape)
    assert fake.count(FAST_F64) == fake.count(FAST_BATCH) == 0
    assert fake.count(GENERAL) == n_general


@pytest.mark.parametrize("case", CASES)
def test_fast_refusal_falls_back_to_the_general_path(fake, case):
    call, entry, n_fast, n_general, check = CASES[case]
    fake.refuse[entry] = n_fast
    check(call(*FAST_SHAPE), *FAST_SHAPE)
    assert fake.count(entry) == n_fast and fake.count(GENERAL) == n_general
    fast_calls = [i for i, (name, _) in enumerate(fake.calls) if name == entry]
    general_calls = [i for i, (name, _) in enumerate(fake.calls) if name == GENERAL]
    assert min(general_calls) > min(fast_calls)
    assert _windows_precede_fast_calls(fake)


def test_a_refusal_of_one_shard_sends_the_whole_batch_to_the_general_path(fake):
    fake.refuse[FAST_BATCH] = 1
    background, ints = _host.separate_batch("original", _batch(*FAST_SHAPE), FAST_SHAPE[0], TUN, devices=[0, 1])
    check_sharded_batch((background, ints), *FAST_SHAPE)
    assert fake.count(FAST_BATCH) == 2 and fake.count(GENERAL) == 3


@pytest.mark.parametrize("status,error", [(_host.REPET_E_TOO_SHORT, ValueError), (_host.REPET_E_INVALID_ARG, ValueError),
                                          (_host.REPET_E_OOM, MemoryError)])
@pytest.mark.parametrize("case", CASES)
def test_other_errors_propagate_without_the_general_path(fake, case, status, error):
    call, entry, _, _, _ = CASES[case]
    fake.fail[entry] = status
    with pytest.raises(error):
        call(*FAST_SHAPE)
    assert fake.count(entry) >= 1 and fake.count(GENERAL) == 0


@pytest.mark.parametrize("case", CASES)
def test_general_path_errors_propagate(fake, case):
    call, _, _, _, _ = CASES[case]
    fake.fail[GENERAL] = _host.REPET_E_TOO_SHORT
    with pytest.raises(ValueError):
        call(96000, 2)
    assert 1 <= fake.count(GENERAL) <= (2 if case == "sharded_track" else 1)  # its two blocks run side by side


def test_malformed_calls_raise_before_any_device_call(fake):
    fs = FAST_SHAPE[0]
    audio = _batch(*FAST_SHAPE)
    with pytest.raises(KeyError):
        _host.separate_batch("original", audio, fs, TUN, in_format="f16")
    with pytest.raises(KeyError):
        _host.separate_batch("original", audio, fs, TUN, out_format="f16")
    for bad in (lambda: _host.separate_batch("median", audio, fs, TUN),
                lambda: _host.driver_batch("median", audio, fs, TUN),
                lambda: _host.separate_f64("median", _clip(*FAST_SHAPE), fs, TUN),
                lambda: _host.separate_batch("original", audio[0], fs, TUN),
                lambda: _host.original_batch(audio[0], fs, TUN),
                lambda: _host.original_batch_pcm16(_pcm(*FAST_SHAPE)[0], fs, TUN),
                lambda: _host.separate_batch("original", audio, fs, TUN, out=np.empty(audio.shape, np.float64)),
                lambda: _host.original_f64(np.zeros(1000), fs, TUN),
                lambda: _host.sim_f64(np.zeros((2, 1000, 2)), fs, TUN)):
        with pytest.raises(ValueError):
            bad()
    assert not [name for name, _ in fake.calls if name in ENTRY_POINTS]


def test_fast_calls_take_the_callers_samples_and_no_by_products(fake):
    """The fast route hands the library the caller's own contiguous samples, and by-product buffers only to
    `separate`."""
    fs, C = FAST_SHAPE
    x = _clip(fs, C)
    _host.sim_f64(x, fs, TUN)
    audio = _batch(fs, C)
    _host.original_batch(audio, fs, TUN)
    (_, f64_args), (_, batch_args) = [call for call in fake.calls if call[0] in (FAST_F64, FAST_BATCH)]
    assert f64_args[2].value == x.ctypes.data and f64_args[7] is None and f64_args[8] is None
    assert batch_args[2].value == audio.ctypes.data


def test_empty_batch(fake):
    background, periods = _host.original_batch(_batch(*FAST_SHAPE, clips=0), FAST_SHAPE[0], TUN)
    assert background.shape == (0, 2, SECONDS * FAST_SHAPE[0]) and periods.shape == (0,)
    background, periods = _host.original_batch(_batch(96000, 2, clips=0), 96000, TUN)
    assert background.shape == (0, 2, SECONDS * 96000) and periods.shape == (0,)
