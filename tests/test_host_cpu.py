"""CPU: the host side of the boundary -- the C-ABI library loads and exports every symbol the
header declares, parameter derivation matches the reference's expressions, the product fails
loudly without a GPU, and the world_size-2 sharding logic works over gloo."""

import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built_library():
    sys.path.insert(0, ROOT)
    import __graft_entry__

    __graft_entry__.build()
    import repet

    return repet._host.load_library()


def test_library_exports_every_declared_symbol(built_library):
    import repet

    header = open(os.path.join(ROOT, "include", "repet_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(repet_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    raw = ctypes.CDLL(repet._host.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), "library does not export %s" % name
        assert name in repet._host.SIGNATURES, "ctypes binding does not cover %s" % name
    assert set(repet._host.SIGNATURES) <= declared
    assert b"sm_100a" in built_library.repet_version()


def test_params_struct_layout_matches_header():
    import repet

    # 12 int32 + 2 doubles, no padding surprises
    assert ctypes.sizeof(repet._host.RepetParams) == 12 * 4 + 2 * 8


@pytest.mark.parametrize(
    "fs,expect",
    [  # SURVEY.md quirk Q16 (banker's rounding at 8/16/32 kHz)
        (8000, (512, 31, 312, 6, 31, 312)),
        (16000, (1024, 31, 312, 6, 31, 312)),
        (22050, (1024, 43, 431, 5, 43, 431)),
        (32000, (2048, 31, 312, 6, 31, 312)),
        (44100, (2048, 43, 431, 5, 43, 431)),
        (48000, (2048, 47, 469, 4, 47, 469)),
        (96000, (4096, 47, 469, 4, 47, 469)),
    ],
)
def test_derived_parameters_follow_the_reference(fs, expect):
    import repet
    import repet_oracle as oracle

    p, window = repet._host.derive_params(fs, repet._tunables())
    got = (p.window_length, p.period_lo, p.period_hi, p.cutoff_bins, p.similarity_distance, p.buffer_frames)
    assert got == expect
    N, w, H = oracle.stft_parameters(fs)
    assert (p.window_length, p.step_length) == (N, H) and np.array_equal(window, w)
    assert p.cola_gain == pytest.approx(1.08, abs=1e-12)
    assert repet._host.number_of_frames(1014301, 2048, 1024) == 992 == oracle.number_of_frames(1014301, 2048, 1024)


def test_module_surface_matches_the_reference():
    import repet

    for name in ("original", "extended", "adaptive", "sim", "simonline", "wavread", "wavwrite", "specshow", "_stft"):
        assert callable(getattr(repet, name))
    defaults = dict(cutoff_frequency=100, period_range=[1, 10], segment_length=10, segment_step=5, filter_order=5,
                    similarity_threshold=0, similarity_distance=1, similarity_number=100, buffer_length=10)
    assert repet._tunables() == defaults  # repet.py:42-63


def test_no_cpu_fallback(built_library):
    """Without a CUDA device the separation call raises; it never routes to the oracle."""
    import repet

    handle = ctypes.c_void_p()
    if built_library.repet_create(0, ctypes.byref(handle)) == 0:
        built_library.repet_destroy(handle)
        pytest.skip("a CUDA device is present")
    with pytest.raises(repet._host.RepetError):
        repet.original(np.zeros((200000, 2)) + 0.1, 44100)
    source = open(os.path.join(ROOT, "repet-python_b200", "repet", "_host.py")).read()
    source += open(os.path.join(ROOT, "repet-python_b200", "repet", "__init__.py")).read()
    assert "repet_oracle" not in source and "import oracle" not in source


def test_wavread_wavwrite_round_trip(tmp_path, wav_pcm):
    import repet

    path = str(tmp_path / "clip.wav")
    repet.wavwrite(wav_pcm[:5000], 44100, path)
    signal, fs = repet.wavread(path)
    assert fs == 44100 and signal.shape == (5000, 2) and signal.dtype == np.float64
    assert np.array_equal(signal, wav_pcm[:5000] / 32768.0)  # repet.py:929


def test_shard_ranges_partition_the_batch():
    from repet_shard import shard_range

    for n in (0, 1, 7, 512, 4096):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(4, 2, 2)


_WORKER = r"""
import os, sys
sys.path.insert(0, os.path.join({root!r}, "oracle")); sys.path.insert(0, os.path.join({root!r}, "repet-python_b200"))
import numpy as np, torch.distributed as dist
import repet_oracle, repet_synth
from repet_shard import shard_range, max_over_ranks, gather_int_arrays
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
lo, hi = shard_range(4, rank, world)
periods = []
for i in range(lo, hi):
    x = repet_synth.make_clip(300 + i, 5 * 44100).T.astype(np.float64)
    periods.append(repet_oracle.original(x, 44100, return_details=True)[1]["period"])
everything = gather_int_arrays(np.array(periods, dtype=np.int32))
slowest = max_over_ranks([10.0 + rank])[0]
if rank == 0:
    print("RESULT", everything.tolist(), slowest)
dist.destroy_process_group()
"""


def test_two_rank_sharding_over_gloo(tmp_path):
    """world_size 2 on CPU: each rank separates its shard (with the oracle standing in for the
    GPU), periods are gathered in rank order, the step time is the max over ranks."""
    import repet_oracle as oracle
    import repet_synth

    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
         "--master-port", "29531", str(script)],
        capture_output=True, text=True, env=env, timeout=300,
    )
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")][0]
    expected = [
        oracle.original(repet_synth.make_clip(300 + i, 5 * 44100).T.astype(np.float64), 44100, return_details=True)[1]["period"]
        for i in range(4)
    ]
    assert line == "RESULT %s 11.0" % expected


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours): one JSON line with the same metric,
    unit and config keys as the CUDA arm, `impl: reference`, a cpu_baseline describing the run and an e2e block
    with zero copy bytes.  One step of one clip per core keeps this to a few seconds."""
    import json
    import subprocess
    import sys

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-sample-clips", "2"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "audio-s/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["n_gpus"] == 1 and line["steps"] == 1
    # the unmodified repet.py where the reference shim finds it, the oracle port everywhere else
    import reference_shim

    expected_kind = "reference" if reference_shim.available() else "port"
    assert line["cpu_baseline"]["kind"] == expected_kind and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


@pytest.mark.parametrize("world", [1, 8])
def test_bench_dump_stays_within_64_mb(tmp_path, world):
    """bench.py --dump-outputs at 512 clips per GPU writes one set of files for the whole run, within 64 MB however
    many GPUs share it, with the backgrounds sampled at fewer positions than a clip has."""
    import bench

    clips, channels, samples = 512 * world, bench.CHANNELS, bench.CLIP_SAMPLES
    positions = bench.dump_positions(clips, channels, samples)
    assert 1 <= len(positions) < samples and np.all(np.diff(positions) > 0) and positions[-1] < samples
    bench.write_dump(str(tmp_path), np.zeros(clips, np.int32), np.zeros((channels, samples), np.float32),
                     np.zeros((clips, channels, len(positions)), np.float32), positions)
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64 << 20


_DUMP_WORKER = r"""
import sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
import bench
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
out = torch.arange(3 * 2 * 5000, dtype=torch.float32).reshape(3, 2, 5000) + 1e5 * rank
periods = torch.arange(3, dtype=torch.int32) + 10 * rank
bench.dump_outputs({directory!r}, torch, dist, world, rank, out, periods)
dist.destroy_process_group()
"""


def test_bench_dump_gathers_every_rank(tmp_path):
    """world_size 2 on CPU: rank 0 writes the clips of both ranks in rank order, once."""
    import bench

    script = tmp_path / "worker.py"
    directory = tmp_path / "dump"
    script.write_text(_DUMP_WORKER.format(root=ROOT, directory=str(directory)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node=2", str(script)],
                         capture_output=True, text=True, env=dict(os.environ, OMP_NUM_THREADS="1"), timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sorted(f.name for f in directory.iterdir()) == [
        "background_clip0.npy", "background_sample.npy", "background_sample_positions.npy", "periods.npy"]
    dumped = {name: np.load(directory / (name + ".npy")) for name in ("periods", "background_clip0", "background_sample",
                                                                      "background_sample_positions")}
    outputs = [np.arange(3 * 2 * 5000, dtype=np.float32).reshape(3, 2, 5000) + 1e5 * rank for rank in range(2)]
    positions = bench.dump_positions(6, 2, 5000)
    assert np.array_equal(dumped["periods"], [0, 1, 2, 10, 11, 12]) and dumped["periods"].dtype == np.float64
    assert np.array_equal(dumped["background_clip0"], outputs[0][0])
    assert np.array_equal(dumped["background_sample_positions"], positions)
    assert np.array_equal(dumped["background_sample"], np.concatenate(outputs)[:, :, positions])


def test_ragged_batches_are_grouped_by_shape_not_padded():
    import repet

    shapes = [(2, 1000), (2, 1200), (2, 1000), (1, 1000), (2, 1200), (2, 1000)]
    groups = repet._host.ragged_groups(shapes)
    assert groups == [((2, 1000), [0, 2, 5]), ((2, 1200), [1, 4]), ((1, 1000), [3])]
    assert sorted(i for _, members in groups for i in members) == list(range(len(shapes)))
    assert repet._host.ragged_groups([]) == []
    with pytest.raises(ValueError):
        repet._host.ragged_groups([(2, 1000, 1)])


def test_shard_bounds_cover_the_batch_in_order():
    """In-process multi-GPU sharding (repet.separate_batch(devices=...)): contiguous, balanced, same split as the
    one-process-per-GPU repet_shard.shard_range."""
    import repet_shard
    from repet import _host

    for n in (0, 1, 7, 8, 512, 4097):
        for g in (1, 2, 3, 8):
            bounds = _host.shard_bounds(n, g)
            assert len(bounds) == g and bounds[0][0] == 0 and bounds[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(bounds, bounds[1:]))
            sizes = [hi - lo for lo, hi in bounds]
            assert max(sizes) - min(sizes) <= 1
            assert [tuple(repet_shard.shard_range(n, r, g)) for r in range(g)] == bounds


def test_param_cache_accepts_array_tunables():
    from repet import _host

    base = dict(cutoff_frequency=100, period_range=[1, 10], segment_length=10, segment_step=5, filter_order=5,
                similarity_threshold=0, similarity_distance=1, similarity_number=100, buffer_length=10)
    p_list, _ = _host.derive_params(44100, base)
    arr = dict(base, period_range=np.array([1, 10]), filter_order=np.int64(5))
    p_arr, _ = _host.derive_params(44100, arr)
    assert (p_arr.period_lo, p_arr.period_hi, p_arr.filter_order) == (p_list.period_lo, p_list.period_hi, p_list.filter_order)
    odd = dict(base, period_range=[[1], [10]])  # nested: still derivable, cached or not
    p_odd, _ = _host.derive_params(44100, odd)
    assert (p_odd.period_lo, p_odd.period_hi) == (p_list.period_lo, p_list.period_hi)


def test_time_blocks_of_one_track_tile_it_on_the_right_grid():
    """repet.extended / adaptive / simonline(devices=...): the cuts of ONE long track (pure host logic)."""
    from repet import _host

    tun = dict(cutoff_frequency=100, period_range=[1, 10], segment_length=10, segment_step=5, filter_order=5,
               similarity_threshold=0, similarity_distance=1, similarity_number=100, buffer_length=10)
    fs = 44100
    for driver, samples in (("extended", 3600 * fs), ("extended", 26 * fs), ("extended", 14 * fs), ("adaptive", 600 * fs),
                            ("adaptive", 100000), ("simonline", 155038 * 1024 + 2048), ("simonline", 12 * fs)):
        params, _ = _host.derive_params(fs, tun, driver)
        for shards in (1, 2, 3, 8):
            blocks = _host.track_time_blocks(driver, samples, params, shards)
            assert 1 <= len(blocks) <= shards
            assert blocks[0][0] == 0 and blocks[-1][1] == samples
            assert all(a[1] == b[0] and a[0] < a[1] for a, b in zip(blocks, blocks[1:]))
            unit = {"extended": params.segment_step, "adaptive": params.segment_step * params.step_length,
                    "simonline": params.step_length}[driver]
            assert all(a % unit == 0 for a, _ in blocks)
    params, _ = _host.derive_params(fs, tun, "extended")
    assert _host.track_time_blocks("extended", 14 * fs, params, 4) == [(0, 14 * fs)]  # a single segment cannot be cut
    params, _ = _host.derive_params(fs, tun, "simonline")
    assert len(_host.track_time_blocks("simonline", 12 * fs, params, 4)) == 1  # the first block needs the warm-up
    with pytest.raises(ValueError):
        _host.track_time_blocks("sim", 10 * fs, params, 2)
