"""GPU: the general-size float64 helper paths (repet_generic.cu) -- _stft / _istft for any window length and step,
_acorr / _beatspectrum for any number of rows (repet.py:1001-1158) -- against the oracle (float64, 1e-10)."""

import numpy as np
import pytest
import scipy.signal.windows

import make_golden
import repet_oracle as oracle
import repet_synth

pytestmark = pytest.mark.gpu

FS = 44100


@pytest.fixture(scope="module")
def repet():
    import repet as module

    module._host.get_handle(0)
    return module


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


@pytest.mark.parametrize("window_length,step_length,samples", [
    (256, 128, 5000),     # the golden helper case of make_golden.helper_inputs (a window no driver uses)
    (256, 64, 5000),      # 75 % overlap: four frames per sample
    (2048, 512, 30000),   # a fast-path length with another hop
    (4096, 2048, 50000),  # 96 kHz window (repet.py:130)
    (8192, 4096, 70000),  # 192 kHz window
    (1000, 300, 12345),   # not a power of two, hop not a divisor: Bluestein
    (255, 100, 4000),     # odd window
    (64, 64, 1000),       # no overlap
    (512, 700, 5000),     # hop longer than the window
])
def test_stft_istft_any_window_and_step(repet, window_length, step_length, samples):
    rng = np.random.default_rng(window_length + step_length)
    x = rng.standard_normal(samples)
    w = scipy.signal.windows.hamming(window_length, sym=False)
    X_ref = oracle.stft(x, w, step_length)
    X = repet._stft(x, w, step_length)
    assert X.shape == X_ref.shape and X.dtype == np.complex128
    assert _rel(X, X_ref) <= 1e-10
    if step_length <= window_length:
        y_ref = oracle.istft(X_ref, w, step_length)
        y = repet._istft(X_ref, w, step_length)
        assert y.shape == y_ref.shape
        assert _rel(y, y_ref) <= 1e-10


def test_stft_golden_helper_vector(repet, golden_helpers):
    """The reference's own outputs for the 256-point helper case (tests/golden/helpers.npz)."""
    h = make_golden.helper_inputs()
    X = repet._stft(h["signal"], h["window"], h["step"])
    assert _rel(X, golden_helpers["stft"]) <= 1e-10
    y = repet._istft(golden_helpers["stft"], h["window"], h["step"])
    assert _rel(y, golden_helpers["istft"]) <= 1e-10


def test_readme_usage_at_96_khz(repet):
    """README.md:79-81 computes abs(repet._stft(mean(x), hamming(N), N/2)) with N from the sampling rate; at 96 kHz
    that is a 4096-point window."""
    fs = 96000
    x = repet_synth.make_clip(31, 3 * fs, 2, fs, 2048).T.astype(np.float64)
    N = pow(2, int(np.ceil(np.log2(0.04 * fs))))
    assert N == 4096
    w = scipy.signal.windows.hamming(N, sym=False)
    spec = np.abs(repet._stft(np.mean(x, axis=1), w, N // 2)[0 : N // 2 + 1, :])
    ref = np.abs(oracle.stft(np.mean(x, axis=1), w, N // 2)[0 : N // 2 + 1, :])
    assert _rel(spec, ref) <= 1e-10


@pytest.mark.parametrize("rows,columns", [(1293, 1025), (3000, 40), (5169, 7), (100, 3)])
def test_acorr_and_beatspectrum_any_size(repet, rows, columns):
    """`repet._beatspectrum(V)` of a 30 s clip (T = 1293 > 1024 frames) used to raise NotImplementedError."""
    rng = np.random.default_rng(rows)
    V = np.abs(rng.standard_normal((columns, rows))) + 0.05 * np.abs(np.sin(np.arange(rows) * 2 * np.pi / 37.0))[None, :]
    b = repet._beatspectrum(V)
    b_ref = oracle.beatspectrum(V)
    assert b.shape == b_ref.shape == (rows,)
    tol = 1e-10 if rows > 1024 else 2e-5  # the small case still goes through the drivers' fp32 beat kernel
    assert _rel(b, b_ref) <= tol
    a = repet._acorr(V.T)
    a_ref = oracle.acorr(V.T)
    assert a.shape == a_ref.shape == (rows, columns)
    assert _rel(a, a_ref) <= (1e-10 if 2 * rows - 1 > 2048 else 2e-5)


def test_beatspectrum_of_a_thirty_second_clip_gives_the_reference_period(repet):
    x = repet_synth.make_clip(11, 30 * FS).astype(np.float64)
    N, w, H = oracle.stft_parameters(FS)
    V = np.stack([np.abs(oracle.stft(x[c], w, H)[: N // 2 + 1]) for c in range(2)], axis=2)
    P = np.power(np.mean(V, axis=2), 2)
    b = repet._beatspectrum(P)
    pr2 = oracle.period_range_frames([1, 10], FS, H)
    assert repet._periods(b, pr2) == oracle.periods(oracle.beatspectrum(P), pr2)


# ---- general float64 DRIVERS (repet_general_f64) -----------------------------------------------------------------
GENERAL_TOL = 1e-9  # float64 end to end: the only differences from the reference are summation orders


@pytest.fixture(scope="module")
def golden_general():
    import os

    return dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "drivers_general.npz")))


def _signal_close(y, y_ref, what, tol=GENERAL_TOL):
    assert y.shape == y_ref.shape, what
    err = float(np.max(np.abs(y - y_ref))) / float(np.max(np.abs(y_ref)))
    assert err <= tol, "%s: max-abs/peak %.3e" % (what, err)


def _general_cases():
    for case, spec in make_golden.GENERAL_CASES.items():
        for fn in spec["functions"]:
            yield case, fn


@pytest.mark.parametrize("case,fn", list(_general_cases()))
def test_general_drivers_match_the_reference(repet, golden_general, case, fn):
    """96 kHz (4096-point window), 192 kHz (8192), 3 / 4 / 5 channels: the reference's outputs recorded by
    oracle/make_golden.py (tests/golden/drivers_general.npz); integers bit-exact, signals to 1e-9 of the peak."""
    import warnings

    warnings.simplefilter("ignore")
    spec = make_golden.GENERAL_CASES[case]
    fs = make_golden.case_fs(spec)
    x = make_golden.case_input(spec)
    key = "%s/%s" % (case, fn)
    tun = repet._tunables()
    if fn == "original":
        y, period = repet._host.original_f64(x, fs, tun, return_period=True)
        assert period == int(golden_general[key + "/period"])
    elif fn == "extended":
        y, periods = repet._host.extended_f64(x, fs, tun, return_periods=True)
        assert np.array_equal(periods, golden_general[key + "/periods"])
    elif fn == "adaptive":
        y, periods = repet._host.adaptive_f64(x, fs, tun, return_periods=True)
        assert np.array_equal(periods, golden_general[key + "/periods"])
    else:
        f = repet._host.sim_f64 if fn == "sim" else repet._host.simonline_f64
        y, lists = f(x, fs, tun, return_indices=True)
        first = int(golden_general.get(key + "/first_frame", 0))
        counts = np.array([len(v) for v in lists[first:]])
        assert np.array_equal(counts, golden_general[key + "/index_counts"])
        assert np.array_equal(np.concatenate(lists[first:]), golden_general[key + "/index_flat"])
    _signal_close(y[:: make_golden.DECIMATE], golden_general[key + "/dec"], key + " (golden)")
    # the drop-in names go the same way
    assert np.array_equal(getattr(repet, fn)(x, fs), y, equal_nan=True)


def test_general_path_agrees_with_the_fast_path_on_a_stereo_clip(repet):
    """The two device implementations against each other where both apply (44.1 kHz stereo): same integers, signals
    within the fast path's fp32 error."""
    x = make_golden.case_input(make_golden.DRIVER_CASES["synth_12s"])
    tun = repet._tunables()
    for method in ("original", "extended", "adaptive", "sim", "simonline"):
        y_general, ints_general = repet._host.general_f64(method, x, FS, tun)
        y_ref = getattr(oracle, method)(x, FS)
        _signal_close(y_general, y_ref, method + " general vs oracle")
        y_fast = getattr(repet, method)(x, FS)
        _signal_close(y_fast, y_general, method + " fast vs general", tol=1e-4)


def test_period_range_above_1024_frames(repet, golden_general):
    """period_range = [1, 30] s is 1292 frames at 44.1 kHz: beyond the fast beat transform, REPET_E_UNSUPPORTED inside,
    the general path outside."""
    spec = make_golden.LONG_PERIOD
    x = repet_synth.make_clip(spec["index"], spec["samples"], spec["channels"]).T.astype(np.float64)
    saved = repet.period_range
    try:
        repet.period_range = list(spec["period_range"])
        y, period = repet._host.original_f64(x, FS, repet._tunables(), return_period=True)
    finally:
        repet.period_range = saved
    assert period == int(golden_general["long_period/original/period"])
    _signal_close(y[:: make_golden.DECIMATE], golden_general["long_period/original/dec"], "long period range")


def test_general_batch_and_separate(repet):
    """Batch and by-product entry points on three-channel clips."""
    audio = repet_synth.make_batch(960, 2, 7 * FS, number_channels=3)
    background, periods = repet.original_batch(audio, FS)
    for i in range(2):
        y_ref, det = oracle.original(audio[i].T.astype(np.float64), FS, return_details=True)
        assert int(periods[i]) == det["period"]
        _signal_close(background[i].T.astype(np.float64), y_ref, "3-channel batch clip %d" % i, tol=1e-6)
    q, _ = repet.separate_batch(audio, FS, "original", out_format="pcm16")
    assert q.shape == (2, 7 * FS, 3) and q.dtype == np.int16
    parts = repet.separate(audio[0].T.astype(np.float64), FS, "adaptive")
    y_ref = oracle.adaptive(audio[0].T.astype(np.float64), FS)
    _signal_close(parts["background"], y_ref, "3-channel separate")
    assert parts["background_spectrogram"].shape == (1025, parts["audio_spectrogram"].shape[1])


def test_stream_at_general_shapes_matches_the_whole_signal_call(repet):
    """repet.SimOnline on a three-channel stream and on a 96 kHz stream: the host-side bookkeeping over windows of
    the general float64 path (ring slots of the whole stream through online_frame_base, quirk Q6)."""
    for fs, channels, seconds in ((FS, 3, 14), (96000, 2, 13)):
        spec = dict(kind="synth", fs=fs, index=970 + channels, samples=seconds * fs + 321, channels=channels)
        x = make_golden.case_input(spec)
        whole = repet.simonline(x, fs)
        stream = repet.SimOnline(fs, channels)
        pieces = [stream.process(x[k : k + fs]) for k in range(0, len(x), fs)]
        pieces.append(stream.flush())
        streamed = np.concatenate(pieces)
        assert streamed.shape == whole.shape
        _signal_close(streamed, whole, "stream %d Hz %d ch" % (fs, channels), tol=1e-12)
        _signal_close(whole, oracle.simonline(x, fs), "whole vs oracle %d Hz %d ch" % (fs, channels))


def test_general_sim_on_a_track_longer_than_one_selection_chunk(repet):
    """The general path's similar-frame selection walks a column in chunks of 4096 frames with halos; a 100 s
    three-channel track (T = 4308) crosses a chunk boundary.  Lists and signal against the oracle."""
    x = repet_synth.make_clip(990, 100 * FS, 3, redraw_seconds=(20, 30)).T.astype(np.float64)
    y, lists = repet._host.sim_f64(x, FS, repet._tunables(), return_indices=True)
    with np.errstate(all="ignore"):
        y_ref, det = oracle.sim(x, FS, return_details=True)
    assert len(lists) == len(det["indices"]) == 4308
    bad = [i for i, (a, b) in enumerate(zip(lists, det["indices"])) if not np.array_equal(a, b)]
    assert not bad, "lists differ at frames %s" % bad[:8]
    _signal_close(y, y_ref, "general sim, 100 s, 3 channels")


def test_batches_fall_back_to_the_general_path_when_the_fast_kernels_refuse(repet):
    """A period range above 1024 frames inside a BATCH call: the fast path answers REPET_E_UNSUPPORTED, the batch
    wrappers route the clips through the general path (the single-clip wrappers already did)."""
    audio = repet_synth.make_batch(995, 2, 90 * FS)
    saved = repet.period_range
    try:
        repet.period_range = [1, 29]  # 1249 frames
        background, periods = repet.original_batch(audio, FS)
        sep, ints = repet.separate_batch(audio, FS, "original")
    finally:
        repet.period_range = saved
    assert np.array_equal(ints[:, 0], periods) and np.array_equal(sep, background)
    for i in range(2):
        y_ref, det = oracle.original(audio[i].T.astype(np.float64), FS, return_details=True, period_range=(1, 29))
        assert int(periods[i]) == det["period"]
        _signal_close(background[i].T.astype(np.float64), y_ref, "clip %d" % i, tol=1e-6)


def test_separate_falls_back_to_the_general_path_when_the_fast_kernels_refuse(repet):
    """`repet.separate` with a period range above 1024 frames: the background, foreground, period and spectrograms
    come from the general path."""
    x = repet_synth.make_batch(995, 1, 90 * FS)[0].T.astype(np.float64)
    saved = repet.period_range
    try:
        repet.period_range = [1, 29]  # 1249 frames
        parts = repet.separate(x, FS)
    finally:
        repet.period_range = saved
    y_ref, det = oracle.original(x, FS, return_details=True, period_range=(1, 29))
    assert parts["integers"].dtype == np.int32 and list(parts["integers"]) == [det["period"]]
    _signal_close(parts["background"], y_ref, "background")
    _signal_close(parts["foreground"], x - y_ref, "foreground", tol=1e-8)
    N, w, H = oracle.stft_parameters(FS)
    for name, signal in (("audio_spectrogram", x), ("background_spectrogram", y_ref), ("foreground_spectrogram", x - y_ref)):
        assert parts[name].dtype == np.float64
        _signal_close(parts[name], np.abs(oracle.stft(np.mean(signal, axis=1), w, H)[: N // 2 + 1]), name, tol=1e-8)


def test_sharded_batch_falls_back_to_the_general_path_when_the_fast_kernels_refuse(repet):
    """`separate_batch(devices=[0])` with a period range above 1024 frames: the shard's refusal sends the batch to
    the general path."""
    audio = repet_synth.make_batch(995, 2, 90 * FS)
    saved = repet.period_range
    try:
        repet.period_range = [1, 29]
        background, ints = repet.separate_batch(audio, FS, "original", devices=[0])
    finally:
        repet.period_range = saved
    assert background.shape == audio.shape and background.dtype == np.float32 and ints.shape == (2, 1)
    for i in range(2):
        y_ref, det = oracle.original(audio[i].T.astype(np.float64), FS, return_details=True, period_range=(1, 29))
        assert int(ints[i, 0]) == det["period"]
        _signal_close(background[i].T.astype(np.float64), y_ref, "clip %d" % i, tol=1e-6)


@pytest.mark.parametrize("fs,channels", [(96000, 2), (FS, 3)])
def test_pcm16_batch_takes_the_general_path(repet, fs, channels):
    """`original_batch_pcm16` at 96 kHz and with three channels: shapes the fast kernels are not compiled for."""
    audio = repet_synth.make_batch(1000 + channels, 2, 8 * fs, channels, fs, step_length=2048 if fs > FS else 1024)
    pcm = np.clip(np.rint(np.transpose(audio, (0, 2, 1)) * 32768.0), -32768, 32767).astype(np.int16)
    background, periods = repet.original_batch_pcm16(pcm, fs)
    assert background.shape == audio.shape and background.dtype == np.float32
    assert periods.shape == (2,) and periods.dtype == np.int32
    for i in range(2):
        y_ref, det = oracle.original(pcm[i] / 32768.0, fs, return_details=True)
        assert int(periods[i]) == det["period"]
        _signal_close(background[i].T.astype(np.float64), y_ref, "%d Hz, %d channels, clip %d" % (fs, channels, i),
                      tol=1e-6)
