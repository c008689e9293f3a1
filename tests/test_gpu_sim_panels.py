"""GPU: repet.sim with the similarity matrix formed in row panels.

A track whose similarity matrix S does not fit the handle's workspace limit is separated panel by panel: the GEMM
writes rows [r0, r0 + P) of S, k_topk settles those columns, and the columns it queues for the exact fallback are
settled once after the last panel.  Every list decision is certified against exact float64 similarities, so panels
must give the same lists, and from them bit-identical backgrounds, as the whole matrix.  Short tracks are forced
through panels with Handle.set_workspace_limit (the panel height follows the limit); the two-hour track needs them
on the default limit."""

import os
import re
import warnings

import numpy as np
import pytest

import make_golden
import make_golden_long
import repet_oracle as oracle
import repet_synth

pytestmark = pytest.mark.gpu

FS = 44100
HOP = 1024
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def repet():
    import repet as module

    module._host.get_handle(0)
    return module


@pytest.fixture(scope="module")
def sm_count():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def _align(v):
    return (v + 255) // 256 * 256


def _linear_bytes(T, nch, number, sm_count):
    """Workspace of one `sim` track besides S, as carve_sim (csrc/repet_drivers.cu) lays it out at 44.1 kHz."""
    xpitch, ppitch, kpad = 1024, 1032, 1056
    b = _align(T * nch * xpitch * 8) + _align(T * ppitch * 4) + _align(T * ppitch * 8) + _align(T * number * 4)
    b += _align(T * 4) + _align(nch * T * ppitch * 4)
    if number > 32:
        b += _align(nch * T * ppitch * 4)
    b += _align(4 * 4)  # k_topk's overflow counters
    return b + 2 * _align(T * kpad * 4) + _align(T * 4) + _align((T * 12 + 255) // 256 * 256 * sm_count * 2)


def _limit_for_rows(T, P, nch, sm_count, number=100):
    """A workspace limit under which S is formed in panels of exactly P rows (P a multiple of 128, P < T)."""
    return _linear_bytes(T, nch, number, sm_count) + 256 + P * T * 4 + 4096


def _frames(n):
    return oracle.number_of_frames(n, 2048, HOP)


def _run(repet, x, handle, limit, capfd=None):
    """sim_f64 on `handle` under `limit`; with capfd also the k_topk statistics (exact-fallback columns, panels)."""
    handle.set_workspace_limit(limit)
    if capfd is not None:
        os.environ["REPET_DEBUG_TOPK"] = "1"
        capfd.readouterr()
    try:
        y, lists = repet._host.sim_f64(x, FS, repet._tunables(), handle=handle, return_indices=True)
    finally:
        handle.set_workspace_limit(0)
        os.environ.pop("REPET_DEBUG_TOPK", None)
    if capfd is None:
        return y, lists, None
    err = capfd.readouterr().err
    m = re.search(r"\((\d+) through the exact fallback\).*; (\d+) row panels of (\d+)", err)
    assert m, err
    return y, lists, tuple(int(g) for g in m.groups())


def _assert_same(lists, y, lists_ref, y_ref, what):
    assert len(lists) == len(lists_ref), what
    bad = [i for i, (a, b) in enumerate(zip(lists, lists_ref)) if not np.array_equal(a, b)]
    assert not bad, "%s: lists differ at frames %s" % (what, bad[:8])
    assert np.array_equal(y, y_ref), "%s: backgrounds differ (max |dy| %.3e)" % (what, float(np.max(np.abs(y - y_ref))))


def _panel_heights(T):
    """128, a height that does not divide T, about T/2, and the largest panel below the whole matrix."""
    odd = next((P for P in range(384, T, 128) if T % P), 128)
    return sorted({128, odd, max(128, (T // 2) // 128 * 128), (T - 1) // 128 * 128})


@pytest.fixture(scope="module")
def inputs(wav_pcm):
    return {
        "sim_long_2min": make_golden.sim_long_input(),
        "wav_full": make_golden.case_input(make_golden.DRIVER_CASES["wav_full"], wav_pcm),
    }


@pytest.mark.parametrize("tensor_core", [2, 1, 0])
@pytest.mark.parametrize("track", ["sim_long_2min", "wav_full"])
def test_panels_equal_the_whole_matrix(repet, inputs, sm_count, capfd, track, tensor_core):
    """Every panel height from 128 to just below T, on each fast pass: same lists, bit-identical background."""
    x = inputs[track]
    T = _frames(len(x))
    handle = repet._host.Handle(0)
    repet._host.set_tuning(simgemm_tc=tensor_core)
    try:
        y_whole, lists_whole, (_, n_whole, _) = _run(repet, x, handle, 0, capfd)
        assert n_whole == 1
        for P in _panel_heights(T):
            y, lists, (_, n_panels, rows) = _run(repet, x, handle, _limit_for_rows(T, P, x.shape[1], sm_count), capfd)
            assert (n_panels, rows) == (-(-T // P), P), (n_panels, rows, P)
            _assert_same(lists, y, lists_whole, y_whole, "%s, simgemm_tc=%d, P=%d" % (track, tensor_core, P))
    finally:
        repet._host.set_tuning(simgemm_tc=2)
        handle.close()
    if track == "sim_long_2min":
        golden = np.load(os.path.join(GOLDEN, "sim_long.npz"))
        assert np.array_equal(np.array([len(v) for v in lists_whole]), golden["counts"].astype(np.int64))
        assert np.array_equal(make_golden.list_digests(lists_whole, make_golden.SIM_LONG["block"]), golden["digests"])


def test_a_limit_below_the_linear_part_gives_128_row_panels(repet, inputs, capfd):
    x = inputs["sim_long_2min"]
    T = _frames(len(x))
    handle = repet._host.Handle(0)
    try:
        y_whole, lists_whole, _ = _run(repet, x, handle, 0)
        y, lists, (_, n_panels, rows) = _run(repet, x, handle, 1 << 20, capfd)
    finally:
        handle.close()
    assert (n_panels, rows) == (-(-T // 128), 128)
    _assert_same(lists, y, lists_whole, y_whole, "1 MB limit")


def test_batches_under_panels_equal_whole_matrix_batches(repet):
    """Three different clips through separate_batch(method="sim") and sim_batch: a panel-forcing limit runs them one
    track per chunk and must give the same integers and backgrounds."""
    audio = repet_synth.make_batch(610, 3, 9 * FS + 311)
    handle = repet._host.get_handle(0)
    bg_whole, ints_whole = repet.separate_batch(audio, FS, method="sim")
    sb_whole, sints_whole = repet.sim_batch(audio, FS)
    handle.set_workspace_limit(1 << 20)
    try:
        bg, ints = repet.separate_batch(audio, FS, method="sim")
        sb, sints = repet.sim_batch(audio, FS)
    finally:
        handle.set_workspace_limit(0)
    # per clip [counts T][indices T x number]: list i is the first counts[i] slots of its row, the rest of the row is
    # not written, so the lists are compared and not the raw rows
    T = _frames(audio.shape[-1])
    for got, ref, what in ((ints, ints_whole, "separate_batch"), (sints, sints_whole, "sim_batch")):
        assert got.shape == ref.shape, what
        for i in range(3):
            assert np.array_equal(got[i, :T], ref[i, :T]), "%s clip %d: list lengths differ" % (what, i)
            lists, lists_ref = repet._host.unpack_lists(got[i], T, 100), repet._host.unpack_lists(ref[i], T, 100)
            bad = [k for k, (a, b) in enumerate(zip(lists, lists_ref)) if not np.array_equal(a, b)]
            assert not bad, "%s clip %d: lists differ at frames %s" % (what, i, bad[:8])
    assert np.array_equal(bg, bg_whole), "separate_batch: backgrounds differ"
    assert np.array_equal(sb, sb_whole), "sim_batch: backgrounds differ"
    assert len({tuple(repet._host.unpack_lists(ints[i], T, 100)[T // 2]) for i in range(3)}) == 3  # different clips


def test_forced_exact_fallback_under_panels_gives_the_golden_lists(repet, inputs, sm_count):
    """Every column queued over all panels, settled once by k_topk_exact after the last one."""
    x = inputs["sim_long_2min"]
    T = _frames(len(x))
    handle = repet._host.Handle(0)
    repet._host.set_tuning(topk_force_exact=1)
    try:
        y, lists, _ = _run(repet, x, handle, _limit_for_rows(T, 1280, x.shape[1], sm_count))
    finally:
        repet._host.set_tuning(topk_force_exact=0)
        handle.close()
    golden = np.load(os.path.join(GOLDEN, "sim_long.npz"))
    assert np.array_equal(np.array([len(v) for v in lists]), golden["counts"].astype(np.int64))
    assert np.array_equal(make_golden.list_digests(lists, make_golden.SIM_LONG["block"]), golden["digests"])
    assert np.all(np.isfinite(y))


def test_stationary_track_under_panels_matches_the_oracle(repet, sm_count, capfd):
    """The near-tied track of test_gpu_sim.py (about T candidates per column) in 384-row panels: its columns still
    overflow the candidate budget, go to the exact fallback, and give the oracle's lists."""
    seconds = 56
    n = seconds * FS
    time = np.arange(n) / FS
    rng = np.random.default_rng(77)
    tone = sum(a * np.sin(2 * np.pi * f * time + p) for a, f, p in ((0.3, 220.0, 0.1), (0.2, 440.0, 1.0), (0.1, 1320.0, 2.0)))
    x = np.stack([tone, 0.8 * tone], axis=1) + 1e-4 * rng.standard_normal((n, 2))
    T = _frames(n)
    handle = repet._host.Handle(0)
    try:
        y, lists, (n_exact, n_panels, rows) = _run(repet, x, handle, _limit_for_rows(T, 384, 2, sm_count), capfd)
    finally:
        handle.close()
    assert rows == 384 and n_panels == -(-T // 384)
    assert n_exact > T // 2
    y_ref, det = oracle.sim(x, FS, return_details=True)
    bad = [i for i, (a, b) in enumerate(zip(lists, det["indices"])) if not np.array_equal(a, b)]
    assert not bad, "lists differ at frames %s" % bad[:8]
    rel = float(np.linalg.norm(y - y_ref) / np.linalg.norm(y_ref))
    assert rel <= 1e-4, rel


def test_ten_minute_golden_through_panels(repet, sm_count, capfd):
    """tests/golden/long_sim_10min.npz (recorded from the reference) in about 8 panels."""
    warnings.simplefilter("ignore")
    path = os.path.join(GOLDEN, "long_sim_10min.npz")
    golden = np.load(path)
    x = make_golden_long.long_input("sim_10min")
    T = _frames(len(x))
    P = -(-T // (8 * 128)) * 128
    handle = repet._host.Handle(0)
    try:
        y, lists, (_, n_panels, rows) = _run(repet, x, handle, _limit_for_rows(T, P, 2, sm_count), capfd)
    finally:
        handle.close()
    assert rows == P and n_panels == 8
    counts = np.array([len(v) for v in lists], dtype=np.int64)
    assert np.array_equal(counts, golden["counts"].astype(np.int64))
    assert np.array_equal(make_golden.list_digests(lists, make_golden_long.BLOCK), golden["digests"])
    dec = y[:: int(golden["decimate"])]
    rel = float(np.linalg.norm(np.ravel(dec - golden["dec"])) / np.linalg.norm(np.ravel(golden["dec"])))
    worst = float(np.max(np.abs(dec - golden["dec"]))) / float(golden["max"])
    assert rel <= 1e-4 and worst <= 1e-4, (rel, worst)


def test_thirty_minutes_whole_and_panels(repet, capfd):
    """30 minutes (T = 77 521): with a 32 GB limit the whole matrix, and the running prune of k_topk keeps every column
    out of the exact fallback; with 8 GB, row panels and the same lists and background."""
    x = repet_synth.make_clip(7330, 1800 * FS, redraw_seconds=(60, 120)).T.astype(np.float64)
    handle = repet._host.Handle(0)
    try:
        y_whole, lists_whole, (n_exact, n_whole, _) = _run(repet, x, handle, 32 << 30, capfd)
        assert n_whole == 1 and n_exact == 0
        y, lists, (n_exact_p, n_panels, _) = _run(repet, x, handle, 8 << 30, capfd)
    finally:
        handle.close()
    assert n_panels > 1 and n_exact_p == 0
    _assert_same(lists, y, lists_whole, y_whole, "30 min, 8 GB limit")


def _stft_frames(x, frames, window):
    """Frames `frames` of oracle.stft of every channel, (N, len(frames), channels) complex128, gathered from the
    samples they cover (centred frames: frame j starts at sample j*H - N/2, zeros outside the signal)."""
    N = len(window)
    idx = np.asarray(frames)[None, :] * HOP - N // 2 + np.arange(N)[:, None]
    inside = (idx >= 0) & (idx < len(x))
    seg = x[np.clip(idx, 0, len(x) - 1)] * inside[:, :, None]
    return np.fft.fft(seg * window[:, None, None], axis=0)


def test_two_hour_track_on_the_default_limit(repet, sm_count, capfd):
    """Two hours (T = 310 080; a whole S would be 385 GB) on the default workspace limit: row panels, no exact
    fallback, workspace within the limit plus the entry point's own staging.  Lists of 64+ frames (seeded ones, the
    first and last frame, the first and last rows of panels 0, 1 and the last) equal oracle.localmaxima of exact
    float64 rows; on 10 s in the middle the background equals the oracle's simmask + _synthesis from those lists."""
    warnings.simplefilter("ignore")
    n = 7200 * FS
    x = repet_synth.make_clip(7200, n, redraw_seconds=(60, 120)).T.astype(np.float64)
    x += 1e-9 * np.random.default_rng(72).standard_normal(x.shape)
    T = _frames(n)
    handle = repet._host.Handle(0)
    try:
        y, lists, (n_exact, n_panels, P) = _run(repet, x, handle, 0, capfd)
        arena = handle.workspace_bytes()
    finally:
        handle.close()
    assert len(lists) == T
    assert n_panels == -(-T // P) and n_panels > 1 and P % 128 == 0
    assert n_exact == 0
    # the workspace: the linear part and one panel of S, within the default limit (at most 24 GiB).  single_f64
    # stages besides it: the lists (T (number + 1) int32), the float64 samples (8 n bytes for n = samples x channels)
    # and three fp32 planes (input, background, foreground: 3 * 4 n bytes)
    samples = n * 2
    staging = _align(T * 101 * 4) + _align(8 * samples) + 3 * _align(4 * samples)
    workspace = _linear_bytes(T, 2, 100, sm_count) + P * T * 4
    assert workspace <= (24 << 30)
    assert arena <= workspace + staging, (arena, workspace, staging)
    # normalised channel-mean magnitude frames with the oracle's STFT convention, chunk by chunk
    N, window, _ = oracle.stft_parameters(FS)
    A = np.empty((T, N // 2 + 1))
    for f0 in range(0, T, 8192):
        f1 = min(T, f0 + 8192)
        V = np.mean(np.abs(_stft_frames(x, np.arange(f0, f1), window)[: N // 2 + 1]), axis=2)
        A[f0:f1] = (V / np.sqrt(np.sum(np.power(V, 2), axis=0))).T
    rng = np.random.default_rng(2)
    frames = {0, T - 1, P - 1, P, 2 * P - 1, (n_panels - 1) * P}
    frames = sorted(frames | set(int(v) for v in rng.integers(0, T, 64)))
    assert len(frames) >= 64
    rows = A @ A[frames].T  # exact float64 similarity rows, one column per frame
    d = int(round(1 * FS / HOP))
    for k, i in enumerate(frames):
        ref = oracle.localmaxima(rows[:, k], 0, d, 100)[1]
        assert np.array_equal(lists[i], ref), "frame %d" % i
    del A, rows
    # background on 10 s in the middle, from the GPU's lists: the window's frames first, then the frames they list
    w0 = T // 2
    w1 = w0 + int(10 * FS / HOP)
    listed = sorted(set().union(*[set(lists[i].tolist()) for i in range(w0, w1)]) - set(range(w0, w1)))
    cols = list(range(w0, w1)) + listed
    pos = {f: k for k, f in enumerate(cols)}
    X = np.concatenate([_stft_frames(x, cols[k : k + 8192], window) for k in range(0, len(cols), 8192)], axis=1)
    local = [np.array([pos[j] for j in lists[i]], dtype=int) for i in range(w0, w1)]
    local += [np.array([], dtype=int)] * len(listed)
    cutoff2 = oracle.cutoff_bins(100, N, FS)
    y_win = y[w0 * HOP : (w1 - 1) * HOP]  # the samples frames w0 .. w1-1 synthesise completely
    for c in range(2):
        mask = oracle.simmask(np.abs(X[: N // 2 + 1, :, c]), local)[:, : w1 - w0]
        ref = oracle._synthesis(mask, X[:, : w1 - w0, c], window, HOP, cutoff2, 10 ** 12)
        got = y_win[:, c]
        assert ref.shape == got.shape
        inner = slice(2 * HOP, len(ref) - 2 * HOP)
        rel = float(np.max(np.abs(got[inner] - ref[inner])) / np.max(np.abs(ref[inner])))
        assert rel <= 1e-4, (c, rel)
