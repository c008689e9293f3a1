"""GPU: the device workspace is sized by the same layout code that carves it.

Every driver lays its buffers out for a chunk of clips and computes its chunk size from that layout measured for
one clip.  Results must not depend on how the workspace limit chunks a batch: at the default limit, at a limit that
leaves room for one clip per chunk, and at 1 MB (one clip per chunk, `sim` in 128-row panels) every driver gives the
same integers and bit-identical backgrounds, through each calling convention.  Every helper entry point must also
run on a fresh handle, whose arena holds only what that helper's own layout asks for."""

import ctypes

import numpy as np
import pytest

import repet_synth

pytestmark = pytest.mark.gpu

FS = 44100
DRIVERS = ["original", "extended", "adaptive", "sim", "simonline"]


@pytest.fixture(scope="module")
def repet():
    import repet as module

    module._host.get_handle(0)
    return module


@pytest.fixture(scope="module")
def inputs():
    """Three 16 s clips (two `extended` segments, longer than simonline's 10 s buffer), and one two-minute clip (many
    `extended` segments), (B, C, S) float32."""
    return {
        "batch": repet_synth.make_batch(420, 3, 16 * FS + 311),
        "long": repet_synth.make_batch(430, 1, 120 * FS + 517),
    }


def _params(repet, handle, driver, number_samples):
    params, _ = repet._host.derive_params(FS, repet._tunables(), driver)
    handle.ensure_window(params.window_length)
    per_clip = int(handle.lib.repet_ints_per_clip(repet._host.METHODS[driver], ctypes.byref(params), number_samples))
    return params, per_clip


def _batch_dev(repet, handle, driver, audio):
    import torch

    n_clips, n_channels, n_samples = audio.shape
    params, per_clip = _params(repet, handle, driver, n_samples)
    x = torch.from_numpy(audio).cuda()
    y = torch.empty_like(x)
    ints = torch.zeros((n_clips, max(1, per_clip)), dtype=torch.int32, device=x.device)
    stream = torch.cuda.current_stream(x.device)
    handle.set_stream(stream.cuda_stream)
    try:
        handle.check(getattr(handle.lib, "repet_%s_batch_dev" % driver)(
            handle.h, ctypes.c_void_p(x.data_ptr()), n_clips, n_channels, n_samples, ctypes.byref(params),
            ctypes.c_void_p(y.data_ptr()), ctypes.c_void_p(ints.data_ptr()), None))
        stream.synchronize()
    finally:
        handle.set_stream(None)
    return y.cpu().numpy(), ints.cpu().numpy()


def _host(fmt):
    def run(repet, handle, driver, audio):
        if fmt == "pcm16":
            audio = np.clip(np.rint(audio.transpose(0, 2, 1) * 32768.0), -32768, 32767).astype(np.int16)
        return repet._host.separate_batch(driver, audio, FS, repet._tunables(), handle=handle, in_format=fmt,
                                          out_format=fmt)
    return run


def _f64(repet, handle, driver, audio):
    """The first clip through repet_<driver>_f64 (float64 (samples, channels))."""
    lib = handle.lib

    def capacity(params, number_samples):
        return int(lib.repet_ints_per_clip(repet._host.METHODS[driver], ctypes.byref(params), number_samples))

    y, ints = repet._host._single_f64_fast("repet_%s_f64" % driver, driver, audio[0].T.astype(np.float64), FS,
                                           repet._tunables(), handle, capacity)
    return y, ints[None, :]


PATHS = {"batch_dev": _batch_dev, "host_f32": _host("f32"), "host_pcm16": _host("pcm16"), "f64": _f64}


def _integers(repet, driver, ints, number):
    """Per clip, the arrays to compare: the periods, or for sim / simonline the counts and the lists (a row's slots
    past its list's count are not written, so the lists are compared and not the raw rows)."""
    if driver not in ("sim", "simonline"):
        return [[row] for row in ints]
    T = ints.shape[1] // (number + 1)
    return [[row[:T]] + repet._host.unpack_lists(row, T, number) for row in ints]


@pytest.mark.parametrize("driver", DRIVERS)
def test_outputs_do_not_depend_on_the_workspace_limit(repet, inputs, driver):
    number = int(repet._tunables()["similarity_number"])
    handle = repet._host.Handle(0)
    try:
        for name, audio in inputs.items():
            # one clip's workspace, measured on a fresh handle: 1.5x of it runs every batch one clip per chunk
            probe = repet._host.Handle(0)
            try:
                _batch_dev(repet, probe, driver, audio[:1])
                one_clip = probe.workspace_bytes() * 3 // 2
            finally:
                probe.close()
            for path, run in PATHS.items():
                ref = None
                for limit in (0, one_clip, 1 << 20):
                    handle.set_workspace_limit(limit)
                    try:
                        y, ints = run(repet, handle, driver, audio)
                    finally:
                        handle.set_workspace_limit(0)
                    got = (y, _integers(repet, driver, ints, number))
                    what = "%s, %s input, %s, limit %d" % (driver, name, path, limit)
                    if ref is None:
                        ref = got
                        continue
                    assert np.array_equal(got[0], ref[0]), what + ": backgrounds differ"
                    assert len(got[1]) == len(ref[1]), what
                    for clip, (a, b) in enumerate(zip(got[1], ref[1])):
                        assert len(a) == len(b) and all(np.array_equal(u, v) for u, v in zip(a, b)), (
                            "%s: integers of clip %d differ" % (what, clip))
    finally:
        handle.close()


def test_every_helper_runs_on_a_fresh_handle(repet):
    host = repet._host
    x = repet_synth.make_clip(440, 7 * FS)
    window = host.hamming_window(2048)
    step = 1024
    spectrum = host.stft_half(x, window, step, handle=host.get_handle(0))
    V = np.abs(spectrum[0]).T.astype(np.float64)  # (1025, T)
    T = V.shape[1]
    lists = host.indices(host.similaritymatrix(V, V, handle=host.get_handle(0)), 0, 3, 40, handle=host.get_handle(0))
    beat = host.beatspectrum(V, handle=host.get_handle(0))
    calls = {
        "stft": lambda h: host.stft_half(x, window, step, handle=h, with_power=True),
        "istft": lambda h: host.istft_half(spectrum, window, step, handle=h),
        "beatspectrum": lambda h: host.beatspectrum(V, handle=h),
        "period": lambda h: host.period_of(V, (1, T // 3), handle=h),
        "mask": lambda h: host.mask(V, 37, handle=h),
        "adaptivemask": lambda h: host.adaptivemask(V, np.full(T, 37), 5, handle=h),
        "beatspectrogram": lambda h: host.beatspectrogram(V, 200, 50, handle=h),
        "selfsimilarity": lambda h: host.selfsimilarity(V, handle=h),
        "periods": lambda h: host.periods(beat, (1, T // 3), handle=h),
        "similarity": lambda h: host.similaritymatrix(V, V[:, 10:15], handle=h),
        "localmaxima": lambda h: host.localmaxima(beat, 0.0, 3, 10, handle=h),
        "simmask": lambda h: host.simmask(V, lists, handle=h),
        "acorr": lambda h: host.acorr(V.T, handle=h),
        "stft_f64": lambda h: host.stft_general(x[0].astype(np.float64), np.hanning(1500), 400, handle=h),
        "istft_f64": lambda h: host.istft_general(host.stft_general(x[0].astype(np.float64), np.hanning(1500), 400,
                                                                    handle=h), np.hanning(1500), 400, handle=h),
        "acorr_f64": lambda h: host.acorr_general(V.T, handle=h),
        "beatspectrum_f64": lambda h: host.beatspectrum_general(V, handle=h),
    }
    for name, call in calls.items():
        handle = host.Handle(0)
        try:
            out = call(handle)
            assert handle.workspace_bytes() > 0, name
        finally:
            handle.close()
        values = out if isinstance(out, tuple) else (out,)
        assert all(np.all(np.isfinite(np.asarray(v))) for v in values), name
