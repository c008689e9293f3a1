"""GPU: the sample formats either side of the separation (repet_separate_batch: fp32 planar or int16 PCM in WAV order,
repet.py:914-946), page-locked host arrays, and the in-process multi-GPU entry point."""

import numpy as np
import pytest

import repet_oracle as oracle
import repet_synth

pytestmark = pytest.mark.gpu

FS = 44100


@pytest.fixture(scope="module")
def repet():
    import repet as module

    module._host.get_handle(0)
    return module


def _valid(repet, method, ints, samples):
    """The integer outputs that carry information: for sim / simonline the [counts][indices] layout leaves the
    slots beyond each list's count unspecified."""
    if method not in ("sim", "simonline"):
        return [ints.tolist()]
    params, _ = repet._host.derive_params(FS, repet._tunables(), method)
    number = params.similarity_number
    frames = ints.shape[1] // (number + 1)
    return [[v.tolist() for v in repet._host.unpack_lists(row, frames, number)] for row in ints]


def _pcm(audio):
    """(B, C, S) float32 -> (B, S, C) int16, the quantisation an int16 WAVE file holds."""
    return np.clip(np.rint(np.transpose(audio, (0, 2, 1)) * 32768.0), -32768, 32767).astype(np.int16)


@pytest.mark.parametrize("method,seconds", [("original", 9), ("extended", 16), ("adaptive", 9), ("sim", 7), ("simonline", 12)])
def test_pcm16_on_either_side_equals_the_fp32_path(repet, method, seconds):
    audio = repet_synth.make_batch(900, 3, seconds * FS + 37)
    pcm = _pcm(audio)
    normalised = np.ascontiguousarray(np.transpose(pcm.astype(np.float32) / 32768.0, (0, 2, 1)))  # repet.py:929
    y32, ints32 = repet.separate_batch(normalised, FS, method)
    # int16 in: the device normalises by 2^15 exactly as above, so the rest of the path sees the same samples
    y_in, ints_in = repet.separate_batch(pcm, FS, method, in_format="pcm16")
    S = audio.shape[2]
    assert _valid(repet, method, ints_in, S) == _valid(repet, method, ints32, S)
    assert np.array_equal(y_in, y32, equal_nan=True)
    # int16 out: round(y * 2^15) to nearest even, saturated, WAV order
    q, ints_q = repet.separate_batch(pcm, FS, method, in_format="pcm16", out_format="pcm16")
    assert q.dtype == np.int16 and q.shape == pcm.shape
    assert _valid(repet, method, ints_q, S) == _valid(repet, method, ints32, S)
    expected = np.clip(np.rint(np.transpose(y32, (0, 2, 1)) * np.float32(32768.0)), -32768, 32767).astype(np.int16)
    assert np.array_equal(q, expected)
    # and against the float64 oracle on the same normalised samples: fp32 path error + 2^-16 of quantisation
    y_ref = getattr(oracle, method)(normalised[0].T.astype(np.float64), FS)
    err = np.max(np.abs(q[0].astype(np.float64) / 32768.0 - y_ref))
    assert err <= 2.0 ** -16 + 1e-4 * np.max(np.abs(y_ref)), err


def test_pcm16_output_saturates(repet):
    audio = repet_synth.make_batch(910, 1, 6 * FS)
    loud = np.ascontiguousarray(audio * (4.0 / np.max(np.abs(audio))))
    y32, _ = repet.separate_batch(loud, FS, "original")
    q, _ = repet.separate_batch(loud, FS, "original", out_format="pcm16")
    assert np.max(np.abs(y32)) > 1.0, "the test input must overdrive the int16 range"
    expected = np.clip(np.rint(np.transpose(y32, (0, 2, 1)) * np.float32(32768.0)), -32768, 32767).astype(np.int16)
    assert np.array_equal(q, expected)
    assert q.max() == 32767 or q.min() == -32768


def test_pinned_arrays_and_in_process_sharding(repet):
    B, S = 5, 8 * FS
    holder_in = repet.pinned_empty((B, 2, S), np.float32)
    holder_out = repet.pinned_empty((B, 2, S), np.float32)
    repet_synth.make_batch(920, B, S, out=holder_in.array)
    y_plain, periods_plain = repet.original_batch(np.array(holder_in.array), FS)
    y, ints = repet.separate_batch(holder_in.array, FS, "original", out=holder_out.array)
    assert y is holder_out.array
    assert np.array_equal(y, y_plain) and np.array_equal(ints[:, 0], periods_plain)
    # one thread + one handle per listed GPU (every visible GPU; a 1-GPU box still goes through the threaded path)
    devices = list(range(repet._host.device_count()))
    y_sharded, periods_sharded = repet.original_batch(holder_in.array, FS, devices=devices)
    assert np.array_equal(y_sharded, y_plain) and np.array_equal(periods_sharded, periods_plain)
    with pytest.raises(ValueError):
        repet.separate_batch(holder_in.array, FS, "original", out=np.empty((B, 2, S), np.float64))
    holder_in.close()
    holder_out.close()


def test_unknown_format_and_method_raise(repet):
    audio = repet_synth.make_batch(930, 1, 5 * FS)
    with pytest.raises(KeyError):
        repet.separate_batch(audio, FS, "original", in_format="f16")
    with pytest.raises(ValueError):
        repet.separate_batch(audio, FS, "median")


def test_numpy_array_tunables(repet):
    """ADVICE r1: a NumPy array tunable (the reference takes np.array(period_range), repet.py:165) must not break the
    parameter cache."""
    x = repet_synth.make_clip(940, 8 * FS).T.astype(np.float64)
    saved = repet.period_range
    try:
        repet.period_range = np.array([1, 10])
        y_arr = repet.original(x, FS)
        repet.period_range = [1, 10]
        y_list = repet.original(x, FS)
    finally:
        repet.period_range = saved
    assert np.array_equal(y_arr, y_list)


def test_istft_selects_its_own_window_length(repet):
    """ADVICE r1: _istft after a driver call at another sampling rate must not transform with the stale window length."""
    rng = np.random.default_rng(5)
    x = rng.standard_normal(6000)
    repet.original(repet_synth.make_clip(941, 6 * 16000, 2, 16000, 512).T.astype(np.float64), 16000)  # leaves N = 1024 set
    import scipy.signal.windows

    w = scipy.signal.windows.hamming(2048, sym=False)
    X = oracle.stft(x, w, 1024)
    y = repet._istft(X, w, 1024)
    y_ref = oracle.istft(X, w, 1024)
    assert y.shape == y_ref.shape
    assert float(np.max(np.abs(y - y_ref))) <= 1e-5 * float(np.max(np.abs(y_ref)))
    # another hop goes through the general float64 path (no longer NotImplementedError)
    X4 = oracle.stft(x, w, 512)
    y4 = repet._istft(X4, w, 512)
    assert float(np.max(np.abs(y4 - oracle.istft(X4, w, 512)))) <= 1e-10


def test_simonline_with_a_ring_longer_than_shared_memory(repet):
    """ADVICE r1: buffer_length above ~16 s (ring of more than 687 frames at 44.1 kHz) used to die with an opaque
    CUDA error; the selection kernel now keeps its similarity rows in global scratch."""
    x = repet_synth.make_clip(942, 24 * FS).T.astype(np.float64)
    saved = repet.buffer_length
    try:
        repet.buffer_length = 20
        y, lists = repet._host.simonline_f64(x, FS, repet._tunables(), return_indices=True)
    finally:
        repet.buffer_length = saved
    y_ref, det = oracle.simonline(x, FS, return_details=True, buffer_length=20)
    first = det["first_frame"]
    assert all(np.array_equal(a, b) for a, b in zip(lists[first:], det["indices"]))
    assert float(np.max(np.abs(y - y_ref))) <= 1e-4 * float(np.max(np.abs(y_ref)))


def test_one_long_track_split_by_time_block(repet):
    """SURVEY.md 8(e) "finer partitions": ONE track cut into time blocks (one per listed device; a repeated device
    runs its blocks in turn, so this also runs on a 1-GPU box) and merged must equal the single-call result."""
    x = repet_synth.make_clip(950, 47 * FS + 777, redraw_seconds=(10, 15)).T.astype(np.float64)
    devices = [0, 0, 0] if repet._host.device_count() < 3 else [0, 1, 2]
    for name, tol in (("extended", 1e-6), ("adaptive", 1e-6), ("simonline", 0.0)):
        whole = getattr(repet, name)(x, FS)
        split = getattr(repet, name)(x, FS, devices=devices)
        assert split.shape == whole.shape
        err = float(np.max(np.abs(split - whole))) / float(np.max(np.abs(whole)))
        assert err <= tol, "%s: %.3e" % (name, err)
    params, _ = repet._host.derive_params(FS, repet._tunables(), "extended")
    assert len(repet._host.track_time_blocks("extended", len(x), params, 3)) == 3


def test_wave_files_in_wave_files_out(repet, tmp_path, wav_pcm):
    """repet.separate_files: int16 WAVE files through the PCM16 batch path (the bundled clip of BASELINE config 1 and
    two synthetic ones of another length), written back as int16; checked against wavread -> original."""
    import scipy.io.wavfile

    clips = {"bundled": wav_pcm[: 9 * FS]}
    for i in range(2):
        audio = repet_synth.make_clip(980 + i, 7 * FS)
        clips["synth%d" % i] = np.clip(np.rint(audio.T * 32768.0), -32768, 32767).astype(np.int16)
    inputs, outputs = [], []
    for name, pcm in clips.items():
        inputs.append(str(tmp_path / (name + ".wav")))
        outputs.append(str(tmp_path / (name + "_background.wav")))
        scipy.io.wavfile.write(inputs[-1], FS, pcm)
    periods = repet.separate_files(inputs, outputs, "original")
    for path_in, path_out, period in zip(inputs, outputs, periods):
        audio_signal, fs = repet.wavread(path_in)
        y_ref, det = oracle.original(audio_signal, fs, return_details=True)
        assert int(period[0]) == det["period"]
        fs_out, written = scipy.io.wavfile.read(path_out)
        assert fs_out == FS and written.dtype == np.int16 and written.shape == y_ref.shape
        err = np.max(np.abs(written / 32768.0 - y_ref))
        assert err <= 2.0 ** -16 + 1e-4 * np.max(np.abs(y_ref)), err


def test_bench_line_contract(repet):
    """bench.py on a small batch: the JSON line carries every key of the contract (roofline, cpu_baseline, e2e with
    its copy bytes, host_link, gpu_launches, clocks, configs)."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--clips-per-gpu", "16", "--steps", "2", "--warmup", "3",
                          "--configs", "cfg1", "--cpu-sample-clips", "2"], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "gpu_launches", "roofline", "cpu_baseline", "e2e",
                "e2e_pcm16", "e2e_numpy_f64", "host_link", "configs"):
        assert key in line, key
    assert line["unit"] == "audio-s/s" and line["scaling"] == "weak" and line["dtype"] == "f32" and line["value"] > 0
    assert line["gpu_launches"] == 7 * line["steps"]
    assert set(line["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and line["roofline"]["bound"] == "hbm"
    assert set(line["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"} and line["cpu_baseline"]["periods_equal_gpu"]
    assert line["e2e"]["h2d_bytes_per_step"] == 16 * 2 * 30 * FS * 4 and line["e2e"]["value"] > 0
    assert line["e2e_pcm16"]["h2d_bytes_per_step"] * 2 == line["e2e"]["h2d_bytes_per_step"]
    assert line["configs"]["cfg1"]["period"] == 286
    assert "workload" in line["config"] and "model" not in line["config"]


def test_bench_dump_outputs(repet, tmp_path):
    """bench.py --dump-outputs: float .npy files of at most 64 MB in all that hold what the last of the --steps timed
    steps returned, with the backgrounds sampled at fewer positions than a clip has.  They are compared with the same
    seeded clips through repet.separate_batch: a check of the dump, not of parity (the golden tests cover that)."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    clips, steps = 8, 3
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--clips-per-gpu", str(clips), "--steps", str(steps),
                          "--warmup", "1", "--configs", "none", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps and line["gpu_launches"] == 7 * steps
    files = sorted(tmp_path.glob("*.npy"))
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    dumped = {f.stem: np.load(f) for f in files}
    assert set(dumped) == {"periods", "background_clip0", "background_sample", "background_sample_positions"}
    assert all(a.dtype in (np.float32, np.float64) for a in dumped.values())
    audio = repet_synth.make_batch(0, clips, 30 * FS)
    background, ints = repet._host.separate_batch("original", audio, FS, repet._tunables())
    assert np.array_equal(dumped["periods"], ints[:, 0])
    assert np.array_equal(dumped["background_clip0"], background[0])
    positions = dumped["background_sample_positions"].astype(np.int64)
    assert len(positions) < 30 * FS
    assert np.array_equal(dumped["background_sample"], background[:, :, positions])
