"""GPU: every median-selection path of the model kernels against np.median, per bin, at chosen list lengths.

k_model (_mask, original / extended), k_adaptive_model and k_adaptive_model_v (_adaptivemask, adaptive) and
k_simmodel / k_simmodel_large / k_simmodel_nyquist (_simmask, sim / simonline) pick a register network, the
-inf/+inf padded 48/64/100/128-slot networks, rank selection or the shared-memory quickselect with a switch on
the list length n.  Here n is chosen to cover every case and every dispatch boundary, at the three bin counts
(257, 513, 1025) and on three kinds of magnitudes: continuous (log-uniform over six decades), heavy ties
(drawn from {0, 1, 2}) and adversarial orderings (ascending, descending, organ-pipe, constant).

Masks are compared per bin, DC and Nyquist included, with the float64 oracle on the fp32-rounded magnitudes
the kernels see.  The bound is relative: the kernels square in fp32 (2^-24), take sqrt.approx (<= 2 ulp), average
the two middles (one rounding), multiply by rsqrt.approx of the fp32 |X|^2 (2^-22.9) and round the mask to fp32,
about 6e-7 in all; RTOL_MASK = 2e-6 holds that with margin, while a neighbouring order statistic of continuous
data is off by orders of magnitude more.  The oracle's eps = 2^-52 (quirk Q10), which the kernels drop, adds up
to eps / (V + eps) on top.
"""

import warnings

import numpy as np
import pytest

import repet_oracle as oracle
import repet_synth

pytestmark = pytest.mark.gpu

FS = 44100
RTOL_MASK = 2e-6
RTOL_SIGNAL = 1e-4
BINS = (257, 513, 1025)
KINDS = ("continuous", "ties", "orderings")


@pytest.fixture(scope="module")
def repet():
    import repet as module

    module._host.get_handle(0)
    return module


def _magnitudes(kind, bins, frames, rng):
    """(bins, frames) float64 magnitudes, already fp32-representable."""
    if kind == "continuous":
        values = np.exp(rng.uniform(np.log(1e-3), np.log(1e3), size=(bins, frames)))
    elif kind == "ties":
        values = rng.integers(0, 3, size=(bins, frames)).astype(np.float64)
    else:  # bins take the four orderings along the frames in turn
        s = np.arange(frames, dtype=np.float64)
        shapes = np.stack([1 + s, frames - s, 1 + np.minimum(s, frames - 1 - s), np.ones(frames)])
        values = np.exp(rng.uniform(-2, 2, size=(bins, 1))) * shapes[np.arange(bins) % 4]
    return values.astype(np.float32).astype(np.float64)


def _assert_mask(got, ref, V, what):
    """Per bin: |got - ref| <= RTOL_MASK |ref| + eps / (V + eps), NaN exactly where the oracle has NaN.
    Returns the largest relative error (eps term removed)."""
    assert got.shape == ref.shape, what
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan), "%s: NaN in %d bins where the oracle has none, or vice versa" % (
        what, int(np.sum(np.isnan(got) != nan)))
    err = np.abs(got - ref)[~nan]
    scale = np.abs(ref[~nan])
    slack = oracle.EPS / (V[~nan] + oracle.EPS)
    bad = err > RTOL_MASK * scale + slack
    if np.any(bad):
        f, t = np.argwhere(~nan)[np.flatnonzero(bad)[0]]
        raise AssertionError("%s: %d bins off, first at bin %d frame %d: %.9g vs oracle %.9g" % (
            what, int(np.sum(bad)), f, t, got[f, t], ref[f, t]))
    with np.errstate(divide="ignore", invalid="ignore"):
        return float(np.max(np.where(scale > 0, np.maximum(err - slack, 0) / scale, 0), initial=0))


def _assert_signal(y, y_ref, what):
    assert y.shape == y_ref.shape, what
    rel = float(np.linalg.norm(np.ravel(y - y_ref)) / max(np.linalg.norm(np.ravel(y_ref)), 1e-300))
    worst = float(np.max(np.abs(y - y_ref)) / max(np.max(np.abs(y_ref)), 1e-300))
    assert rel <= RTOL_SIGNAL and worst <= RTOL_SIGNAL, "%s: rel L2 %.3e, max-abs/max %.3e" % (what, rel, worst)
    print("%s: rel L2 %.2e, max-abs/max %.2e" % (what, rel, worst))


# ---- _simmask: k_simmodel, k_simmodel_large, k_simmodel_nyquist ----------------------------------------
SOURCES = 240
LONGEST = 219  # the longest list the shared-memory median of k_simmodel holds (launch_simmodel's budget)


def _simmask_case(kind, bins, rng):
    """Source frames carry the data; target frame SOURCES + n gets a list of n sources (n = 0..LONGEST) and a
    magnitude ~1e3 x the largest source in every bin, so that its mask is model / V: the median itself."""
    sources = _magnitudes(kind, bins, SOURCES, rng)
    peak = np.max(sources, axis=1, keepdims=True)
    targets = 1e3 * np.where(peak > 0, peak, 1.0) * rng.uniform(1, 2, size=(bins, LONGEST + 1))
    V = np.concatenate([sources, targets], axis=1).astype(np.float32).astype(np.float64)
    # the sources' own lists are short (register networks, and the min with their own magnitude)
    lists = [np.sort(rng.choice(SOURCES, size=(7 * i) % 33, replace=False)) for i in range(SOURCES)]
    for n in range(LONGEST + 1):
        members = np.sort(rng.choice(SOURCES, size=n, replace=False))  # ascending frames: sorted for "orderings"
        if n % 3 == 1:
            members = members[::-1]
        if n >= 2 and n % 5 == 0:
            members[rng.integers(n)] = members[rng.integers(n)]  # a frame listed twice
        lists.append(members)
    return V, lists


def _simmask_oracle(V, lists):
    with warnings.catch_warnings():  # np.median of the empty list: NaN and a RuntimeWarning, as in the reference
        warnings.simplefilter("ignore", RuntimeWarning)
        return oracle.simmask(V, lists)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("bins", BINS)
def test_simmask_every_list_length(repet, bins, kind):
    rng = np.random.default_rng(100 * bins + KINDS.index(kind))
    V, lists = _simmask_case(kind, bins, rng)
    M = repet._simmask(V, lists)
    ref = _simmask_oracle(V, lists)
    assert np.all(np.isnan(M[:, SOURCES])), "an empty list gives a NaN column, as np.median([]) does"
    worst = _assert_mask(M, ref, V, "_simmask %d bins, %s (target frame %d has the list of length 0)" % (
        bins, kind, SOURCES))
    print("_simmask %4d bins %-10s: max relative error %.2e" % (bins, kind, worst))


def test_simmask_refuses_a_list_longer_than_the_shared_memory_median(repet):
    rng = np.random.default_rng(7)
    V, lists = _simmask_case("continuous", 1025, rng)
    too_long = list(lists)
    too_long[-1] = np.arange(LONGEST + 1) % SOURCES
    with pytest.raises(NotImplementedError):
        repet._simmask(V, too_long)
    # the refusal leaves the handle usable
    _assert_mask(repet._simmask(V, lists), _simmask_oracle(V, lists), V, "_simmask after a refused call")


# ---- _mask: k_model ------------------------------------------------------------------------------------
# (r, p): T = (r - 1) p + k0 with 0 < k0 < p, so phases q < k0 take r frames and the others r - 1.  Together
# the counts cover 1..41: networks up to 32, rank selection above.  p = 1 (every phase takes r), p < 8, p not a
# multiple of MODEL_QB = 8, and p > 128 (the Nyquist CTA loops over phases 128 apart).
MASK_SHAPES = [(2, 3), (4, 5), (6, 7), (8, 13), (10, 130), (12, 2), (14, 9), (16, 6), (18, 11), (20, 150), (22, 3),
               (24, 17), (26, 5), (28, 7), (30, 10), (32, 131), (34, 4), (36, 12), (38, 9), (40, 3), (41, 2),
               (5, 1), (33, 1)]


def _mask_frames(r, p):
    return r if p == 1 else (r - 1) * p + (p + 1) // 2


def test_mask_shapes_cover_every_count():
    counts = set()
    for r, p in MASK_SHAPES:
        T = _mask_frames(r, p)
        counts |= {len(range(q, T, p)) for q in range(p)}
    assert counts >= set(range(1, 42))
    assert any(p == 1 for _, p in MASK_SHAPES) and any(p > 128 for _, p in MASK_SHAPES)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("bins", BINS)
def test_mask_every_count_per_phase(repet, bins, kind):
    rng = np.random.default_rng(200 * bins + KINDS.index(kind))
    worst = 0.0
    for r, p in MASK_SHAPES:
        V = _magnitudes(kind, bins, _mask_frames(r, p), rng)
        worst = max(worst, _assert_mask(repet._mask(V, p), oracle.mask(V, p), V, "_mask %d bins, %s, r=%d p=%d" % (
            bins, kind, r, p)))
    print("_mask %4d bins %-10s: max relative error %.2e" % (bins, kind, worst))


# ---- _adaptivemask: k_adaptive_model (the spectra path) ------------------------------------------------
ADAPTIVE_FRAMES = 150


def _adaptive_periods(rng):
    """Per-frame periods: 1, small, near T, >= T and random, so that the in-range count of every frame is clipped
    to each value from 1 to the filter order somewhere."""
    T = ADAPTIVE_FRAMES
    periods = rng.integers(1, T + 6, size=T)
    periods[::9] = 1
    periods[4::9] = rng.integers(2, 8, size=len(periods[4::9]))
    periods[2::13] = T - 1
    periods[6::17] = T + 3
    periods[60:80] = T // np.arange(1, 21)  # about k of the offsets in range, around the middle frames
    periods[100:120] = T // np.arange(1, 21) + 1
    return periods


def _adaptive_counts(periods, order):
    T = len(periods)
    offsets = np.arange(1, order + 1) - int(np.ceil(order / 2))
    return np.array([np.sum((i + offsets * periods[i] >= 0) & (i + offsets * periods[i] < T)) for i in range(T)])


def test_adaptive_periods_cover_every_count():
    periods = _adaptive_periods(np.random.default_rng(0))
    for order in range(1, 21):
        assert set(_adaptive_counts(periods, order)) == set(range(1, order + 1)), order


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("bins", BINS)
def test_adaptivemask_every_count(repet, bins, kind):
    rng = np.random.default_rng(300 * bins + KINDS.index(kind))
    periods = _adaptive_periods(np.random.default_rng(0))
    worst = 0.0
    for order in range(1, 21):  # register networks up to 16, rank selection above
        V = _magnitudes(kind, bins, ADAPTIVE_FRAMES, rng)
        M = repet._adaptivemask(V, periods, order)
        ref = oracle.adaptivemask(V, periods, order)
        worst = max(worst, _assert_mask(M, ref, V, "_adaptivemask %d bins, %s, order %d" % (bins, kind, order)))
    print("_adaptivemask %4d bins %-10s: max relative error %.2e" % (bins, kind, worst))


# ---- the adaptive driver on both model kernels ---------------------------------------------------------
ADAPTIVE_TUNABLES = dict(period_range=[0.1, 0.4], segment_length=4, segment_step=2)


@pytest.fixture(scope="module")
def adaptive_clip():
    return _adaptive_clip()


def _adaptive_clip():
    """8 s of stereo under an envelope that repeats every 10 frames: a DC offset, a +-1 alternation (the
    Nyquist bin) and a repeating noise burst, different per channel, plus a little fresh noise."""
    rng = np.random.default_rng(2024)
    n = 8 * FS
    period = 10 * 1024
    i = np.arange(n)
    envelope = 0.3 + 0.7 * (0.5 + 0.5 * np.cos(2 * np.pi * i / period)) ** 2
    alternation = np.where(i % 2 == 0, 1.0, -1.0)
    burst = np.tile(rng.standard_normal((2, period)), (1, n // period + 1))[:, :n]
    channels = [envelope * (dc + ny * alternation + 0.2 * burst[c]) + 0.02 * rng.standard_normal(n)
                for c, (dc, ny) in enumerate(((0.3, 0.2), (-0.2, 0.25)))]
    return np.stack(channels, axis=1)


@pytest.mark.parametrize("order", range(1, 17))
def test_adaptive_driver_both_model_kernels(repet, adaptive_clip, order):
    """adaptive_vsq = 1 runs k_adaptive_model_v on the |X|^2 planes of k_stft, 0 runs k_adaptive_model on the
    spectra.  Only the right channel's |X|^2 can differ between them, in the last bit (fma operand order: k_stft
    squares a - conj(b), the spectra hold it rotated), and since one complex inverse transform carries both
    channels, that reaches both outputs: the two must agree to ~1e-7 of the peak, far below any median error."""
    x = adaptive_clip
    tunables = dict(ADAPTIVE_TUNABLES, filter_order=order)
    saved = {name: getattr(repet, name) for name in tunables}
    results = {}
    try:
        for name, value in tunables.items():
            setattr(repet, name, value)
        for vsq in (1, 0):
            repet._host.set_tuning(adaptive_vsq=vsq)
            results[vsq] = repet._host.adaptive_f64(x, FS, repet._tunables(), return_periods=True)
    finally:
        repet._host.set_tuning(adaptive_vsq=1)
        for name, value in saved.items():
            setattr(repet, name, value)
    y_ref, det = oracle.adaptive(x, FS, return_details=True, **tunables)
    periods = np.asarray(det["periods"])
    counts = _adaptive_counts(periods, order)
    assert counts.max() == order and (order == 1 or counts.min() < order)  # the full count, and clipped ones at the edges
    for vsq, (y, got) in results.items():
        assert np.array_equal(got, periods), "adaptive_vsq=%d: per-frame periods" % vsq
        _assert_signal(y, y_ref, "adaptive order %d, adaptive_vsq=%d" % (order, vsq))
    (y1, _), (y0, _) = results[1], results[0]
    gap = float(np.max(np.abs(y1 - y0)) / np.max(np.abs(y0)))
    print("adaptive order %2d: |vsq - spectra| max-abs/peak %.2e" % (order, gap))
    assert gap <= 1e-6


# ---- the sim driver at the dispatch boundaries -----------------------------------------------------------
@pytest.fixture(scope="module")
def sim_clip():
    return _sim_clip()


def _sim_clip():
    x = repet_synth.make_clip(4242, 6 * FS).T.astype(np.float64)  # T = 260 frames
    assert oracle.number_of_frames(len(x), 2048, 1024) == 260
    return x


@pytest.mark.parametrize("number", [32, 33, 48, 49, 64, 65, 100, 101, 128, 129, 219, 220])
def test_sim_driver_list_lengths_at_the_boundaries(repet, sim_clip, number):
    """similarity_distance = 0 and threshold 0: every frame is a candidate, so every list holds exactly
    `number` frames -- both sides of each k_simmodel / k_simmodel_large / k_simmodel_nyquist branch, on two
    interleaved channels.  220 is over the shared-memory budget: the fast path refuses and the general path
    gives the same result."""
    x = sim_clip
    tunables = dict(similarity_distance=0, similarity_number=number)
    saved = {name: getattr(repet, name) for name in tunables}
    try:
        for name, value in tunables.items():
            setattr(repet, name, value)
        tun = repet._tunables()
        y, lists = repet._host.sim_f64(x, FS, tun, return_indices=True)
        if number > LONGEST:
            handle = repet._host.get_handle(0)
            with pytest.raises(NotImplementedError):
                repet._host._single_f64_fast("repet_sim_f64", "sim", x, FS, tun, handle,
                                             lambda params, samples: 260 * (number + 1))
    finally:
        for name, value in saved.items():
            setattr(repet, name, value)
    y_ref, det = oracle.sim(x, FS, return_details=True, **tunables)
    assert all(len(v) == number for v in det["indices"])
    assert len(lists) == len(det["indices"])
    bad = [i for i, (a, b) in enumerate(zip(lists, det["indices"])) if not np.array_equal(a, b)]
    assert not bad, "lists differ at frames %s" % bad[:8]
    _assert_signal(y, y_ref, "sim, similarity_number %d" % number)
