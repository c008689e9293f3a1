"""GPU: repet.sim on the general float64 path with the similarity matrix formed in row panels.

Inputs the fast path does not take (sampling rates above 51.2 kHz, more than two channels) run repet_general_f64.  Its
`sim` forms S = An An^T in float64 with one fma chain per element over ascending k, so S is bitwise symmetric and a
panel of rows [r0, r0 + P) holds exactly the columns whose lists it settles.  When S and the selection scratch,
need(P) = P T 8 + min(P, 2 SMs) T 4 bytes, do not fit the handle's workspace limit for P = T, S is formed in panels of
the largest multiple of 64 rows that fits.  Panels must give the whole matrix's lists and bit-identical backgrounds.
Each Gram + selection pair adds two to the handle's launch count, which tells how many panels a call formed."""

import ctypes
import os
import warnings

import numpy as np
import pytest

import make_golden
import repet_oracle as oracle
import repet_synth

pytestmark = pytest.mark.gpu

FS96 = 96000
HOP96 = 2048
NUMBER = 100  # similarity_number
GOLDEN_SIM_CASES = ["synth96k_13s", "synth192k_5s", "synth44k_3ch_12s", "synth44k_5ch_8s"]


@pytest.fixture(scope="module")
def repet():
    import repet as module

    module._host.get_handle(0)
    return module


@pytest.fixture(scope="module")
def sm_count():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def golden_general():
    return dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "drivers_general.npz")))


def _need(P, T, sm_count):
    """Bytes of one S panel of P rows and of k_gen_indices' per-CTA kept lists (gen_run in csrc/repet_generic.cu)."""
    return P * T * 8 + min(P, 2 * sm_count) * T * 4


def _panel_rows(T, limit, sm_count):
    """The panel height gen_run picks under `limit`: T when need(T) fits, else the largest multiple of 64 that fits
    (64 at least)."""
    if _need(T, T, sm_count) <= limit:
        return T
    P = min(T, limit // (T * 8)) // 64 * 64
    while P > 64 and _need(P, T, sm_count) > limit:
        P -= 64
    return min(T, max(P, 64))


def _panel_heights(T):
    """64, a height that does not divide T, about T/2, and the largest multiple of 64 below T."""
    odd = next((P for P in range(192, T, 64) if T % P), 64)
    half = min(max(64, int(round(T / 2 / 64)) * 64), (T - 1) // 64 * 64)
    return sorted({64, odd, half, (T - 1) // 64 * 64})


def _frames(n, fs):
    N, _, H = oracle.stft_parameters(fs)
    return oracle.number_of_frames(n, N, H)


def _sim(repet, x, fs, handle, limit):
    """sim_f64 on `handle` under `limit` (0: the default); returns (background, lists, launches of the call)."""
    handle.set_workspace_limit(limit)
    try:
        before = handle.launch_count()
        y, lists = repet._host.sim_f64(x, fs, repet._tunables(), handle=handle, return_indices=True)
        launches = handle.launch_count() - before
    finally:
        handle.set_workspace_limit(0)
    return y, lists, launches


def _assert_same(lists, y, lists_ref, y_ref, what):
    assert len(lists) == len(lists_ref), what
    bad = [i for i, (a, b) in enumerate(zip(lists, lists_ref)) if not np.array_equal(a, b)]
    assert not bad, "%s: lists differ at frames %s" % (what, bad[:8])
    assert np.array_equal(y, y_ref, equal_nan=True), "%s: backgrounds differ" % what


@pytest.mark.parametrize("case", GOLDEN_SIM_CASES)
def test_golden_lists_under_panels(repet, golden_general, sm_count, case):
    """The four general `sim` goldens (96 and 192 kHz, 3 and 5 channels) at panel heights from 64 to just below T:
    the golden lists, and the background of the default limit bit for bit."""
    warnings.simplefilter("ignore")
    spec = make_golden.GENERAL_CASES[case]
    fs = make_golden.case_fs(spec)
    x = make_golden.case_input(spec)
    T = _frames(len(x), fs)
    key = "%s/sim" % case
    handle = repet._host.Handle(0)
    try:
        y_whole, lists_whole, launches_whole = _sim(repet, x, fs, handle, 0)
        for P in _panel_heights(T):
            limit = _need(P, T, sm_count)
            assert _panel_rows(T, limit, sm_count) == P
            y, lists, launches = _sim(repet, x, fs, handle, limit)
            what = "%s, P=%d" % (case, P)
            assert launches - launches_whole == 2 * (-(-T // P) - 1), what  # one Gram + one selection per panel
            assert np.array_equal([len(v) for v in lists], golden_general[key + "/index_counts"]), what
            assert np.array_equal(np.concatenate(lists), golden_general[key + "/index_flat"]), what
            _assert_same(lists, y, lists_whole, y_whole, what)
    finally:
        handle.close()


def test_silent_stretch_under_panels(repet, sm_count):
    """A 96 kHz clip with 3 s of digital silence (quirk Q18): the all-zero frames have NaN rows of S, empty lists and
    a NaN background; panels reproduce the whole matrix's output exactly, NaN for NaN."""
    warnings.simplefilter("ignore")
    x = repet_synth.make_clip(1801, 12 * FS96 + 77, 2, FS96, HOP96).T.astype(np.float64)
    x[4 * FS96 : 7 * FS96] = 0.0
    T = _frames(len(x), FS96)
    handle = repet._host.Handle(0)
    try:
        y_whole, lists_whole, launches_whole = _sim(repet, x, FS96, handle, 0)
        silent = [i for i in range(T) if len(lists_whole[i]) == 0]
        assert len(silent) > 100, len(silent)
        assert np.isnan(y_whole[5 * FS96]).all() and np.isfinite(y_whole[FS96]).all()
        for P in (64, 192):
            y, lists, launches = _sim(repet, x, FS96, handle, _need(P, T, sm_count))
            assert launches - launches_whole == 2 * (-(-T // P) - 1), P
            _assert_same(lists, y, lists_whole, y_whole, "silent stretch, P=%d" % P)
    finally:
        handle.close()


CU_MEMPOOL_ATTR_USED_MEM_HIGH = 8  # cuda.h, enum CUmemPool_attribute


def _default_pool_used_high(reset):
    """High-water mark of the device's default memory pool (what cudaMallocAsync draws from), through the driver API;
    `reset` sets it back to what is in use now."""
    cuda = ctypes.CDLL("libcuda.so.1")
    assert cuda.cuInit(0) == 0
    device = ctypes.c_int()
    assert cuda.cuDeviceGet(ctypes.byref(device), 0) == 0
    pool = ctypes.c_void_p()
    assert cuda.cuDeviceGetDefaultMemPool(ctypes.byref(pool), device) == 0
    value = ctypes.c_uint64(0)
    if reset:
        assert cuda.cuMemPoolSetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_HIGH, ctypes.byref(value)) == 0
    assert cuda.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_HIGH, ctypes.byref(value)) == 0
    return value.value


def test_the_workspace_limit_bounds_the_similarity_matrix(repet, sm_count):
    """10 minutes at 96 kHz mono (T = 28 126, whole S = 6.3 GB) under a 1 GiB limit: the device memory the call takes
    from the pool peaks at the linear buffers plus at most 1 GiB, and the output is that of the default limit."""
    warnings.simplefilter("ignore")
    n, C = 600 * FS96, 1
    x = repet_synth.make_clip(1802, n, C, FS96, HOP96, redraw_seconds=(60, 120)).T.astype(np.float64)
    N, _, _ = oracle.stft_parameters(FS96)
    F = N // 2 + 1
    T = _frames(n, FS96)
    assert T == 28126
    limit = 1 << 30
    P = _panel_rows(T, limit, sm_count)
    assert P < T
    # repet_general_f64: audio, background, window, ints; gen_run: X and tmp (C T N complex128), V (C T F), Vm, An
    linear = 2 * n * C * 8 + N * 8 + T * (NUMBER + 1) * 4 + 2 * C * T * N * 16 + C * T * F * 8 + 2 * T * F * 8
    slack = 256 << 20  # the pool's rounding of the call's dozen allocations
    handle = repet._host.Handle(0)
    try:
        _default_pool_used_high(reset=True)
        y, lists, launches = _sim(repet, x, FS96, handle, limit)
        peak = _default_pool_used_high(reset=False)
        y_whole, lists_whole, launches_whole = _sim(repet, x, FS96, handle, 0)
    finally:
        handle.close()
    assert peak <= linear + _need(P, T, sm_count) + slack, (peak, linear, P)
    assert peak <= linear + limit + slack
    assert launches - launches_whole == 2 * (-(-T // P) - 1)
    _assert_same(lists, y, lists_whole, y_whole, "10 min, 1 GiB limit")


def test_batch_fallback_honours_the_handle_limit(repet, sm_count):
    """separate_batch(method="sim") on three 96 kHz clips goes clip by clip through the general path on the process
    handle; a limit that forces 128-row panels there gives the default limit's lists and backgrounds."""
    warnings.simplefilter("ignore")
    audio = repet_synth.make_batch(1803, 3, 9 * FS96 + 500, 2, FS96, step_length=HOP96)
    T = _frames(audio.shape[-1], FS96)
    handle = repet._host.get_handle(0)
    before = handle.launch_count()
    bg_whole, ints_whole = repet.separate_batch(audio, FS96, method="sim")
    launches_whole = handle.launch_count() - before
    handle.set_workspace_limit(_need(128, T, sm_count))
    try:
        before = handle.launch_count()
        bg, ints = repet.separate_batch(audio, FS96, method="sim")
        launches = handle.launch_count() - before
    finally:
        handle.set_workspace_limit(0)
    assert launches - launches_whole == 3 * 2 * (-(-T // 128) - 1)
    assert ints.shape == ints_whole.shape
    for i in range(3):
        lists = repet._host.unpack_lists(ints[i], T, NUMBER)
        lists_ref = repet._host.unpack_lists(ints_whole[i], T, NUMBER)
        bad = [k for k, (a, b) in enumerate(zip(lists, lists_ref)) if not np.array_equal(a, b)]
        assert not bad, "clip %d: lists differ at frames %s" % (i, bad[:8])
    assert np.array_equal(bg, bg_whole)


def _stft_frames(x, frames, window):
    """Frames `frames` of oracle.stft of every channel at 96 kHz, (N, len(frames), channels) complex128, gathered
    from the samples they cover (centred frames: frame j starts at sample j*H - N/2, zeros outside the signal)."""
    N = len(window)
    idx = np.asarray(frames)[None, :] * HOP96 - N // 2 + np.arange(N)[:, None]
    inside = (idx >= 0) & (idx < len(x))
    seg = x[np.clip(idx, 0, len(x) - 1)] * inside[:, :, None]
    return np.fft.fft(seg * window[:, None, None], axis=0)


def test_one_hour_at_96_khz_on_the_default_limit(repet, sm_count):
    """One hour at 96 kHz mono (T = 168 751; a whole S would be 228 GB) on the default workspace limit (24 GiB on an
    idle B200): row panels.  Lists of 64+ frames (seeded ones, the first and last frame, and the first and last rows
    of panels 0, 1 and the last for the 24 GiB panel height) equal oracle.localmaxima of exact float64 rows; on 10 s
    in the middle the background equals the oracle's simmask + _synthesis from those lists."""
    warnings.simplefilter("ignore")
    n = 3600 * FS96
    x = repet_synth.make_clip(1804, n, 1, FS96, HOP96, redraw_seconds=(60, 120)).T.astype(np.float64)
    x += 1e-9 * np.random.default_rng(96).standard_normal(x.shape)  # no two similarities tie exactly
    T = _frames(n, FS96)
    assert T == 168751
    handle = repet._host.Handle(0)
    try:
        # the launches of a call with a single Gram + selection pair, from a short clip
        _, _, launches_one = _sim(repet, x[: 20 * FS96], FS96, handle, 0)
        y, lists, launches = _sim(repet, x, FS96, handle, 0)
    finally:
        handle.close()
    assert len(lists) == T
    n_panels = 1 + (launches - launches_one) // 2
    P = _panel_rows(T, 24 << 30, sm_count)
    assert n_panels >= -(-T // P) > 1, (n_panels, P)
    N, window, _ = oracle.stft_parameters(FS96)
    A = np.empty((T, N // 2 + 1))
    for f0 in range(0, T, 4096):
        f1 = min(T, f0 + 4096)
        V = np.mean(np.abs(_stft_frames(x, np.arange(f0, f1), window)[: N // 2 + 1]), axis=2)
        A[f0:f1] = (V / np.sqrt(np.sum(np.power(V, 2), axis=0))).T
    rng = np.random.default_rng(3)
    last = (-(-T // P) - 1) * P
    frames = {0, T - 1, P - 1, P, 2 * P - 1, last - 1, last}
    frames = sorted(frames | set(int(v) for v in rng.integers(0, T, 64)))
    assert len(frames) >= 64
    rows = A @ A[frames].T  # exact float64 similarity rows, one column per frame
    d = int(round(1 * FS96 / HOP96))
    for k, i in enumerate(frames):
        ref = oracle.localmaxima(rows[:, k], 0, d, NUMBER)[1]
        assert np.array_equal(lists[i], ref), "frame %d" % i
    del A, rows
    # background on 10 s in the middle, from the GPU's lists: the window's frames first, then the frames they list
    w0 = T // 2
    w1 = w0 + int(10 * FS96 / HOP96)
    listed = sorted(set().union(*[set(lists[i].tolist()) for i in range(w0, w1)]) - set(range(w0, w1)))
    cols = list(range(w0, w1)) + listed
    pos = {f: k for k, f in enumerate(cols)}
    X = np.concatenate([_stft_frames(x, cols[k : k + 4096], window) for k in range(0, len(cols), 4096)], axis=1)
    local = [np.array([pos[j] for j in lists[i]], dtype=int) for i in range(w0, w1)]
    local += [np.array([], dtype=int)] * len(listed)
    cutoff2 = oracle.cutoff_bins(100, N, FS96)
    mask = oracle.simmask(np.abs(X[: N // 2 + 1, :, 0]), local)[:, : w1 - w0]
    ref = oracle._synthesis(mask, X[:, : w1 - w0, 0], window, HOP96, cutoff2, 10 ** 12)
    got = y[w0 * HOP96 : (w1 - 1) * HOP96, 0]  # the samples frames w0 .. w1-1 synthesise completely
    assert ref.shape == got.shape
    inner = slice(2 * HOP96, len(ref) - 2 * HOP96)
    rel = float(np.max(np.abs(got[inner] - ref[inner])) / np.max(np.abs(ref[inner])))
    assert rel <= 1e-9, rel
