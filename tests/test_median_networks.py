"""CPU: the generated median-selection networks (repet-python_b200/csrc/median_networks*.cuh), read back from
the headers the kernels compile and executed statement by statement.

* The headers are what tools/gen_median_networks.py emits for n = 1..32 and 48/64/100/128.
* n = 1..32: both middle outputs, (n-1)//2 and n//2, are right on every one of the 2^n inputs of 0s and 1s.
  The networks are built from min and max only, so they commute with every monotone map; by the zero-one
  principle that proves them right on all real inputs.  The check is independent of the generator's own
  `verify` (which samples 0/1 placements above n = 22).
* n = 33..128: padded exactly as gather_median_large pads a similar-frame list, (NS - n) >> 1 slots of -inf
  and the rest +inf, the NS-slot network the kernels dispatch to leaves np.median's order statistics in
  v[NS/2 - 1] (and v[NS/2]).
"""

import importlib.util
import os
import re
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "repet-python_b200", "csrc")
TMP = -1  # the scratch register `t` of a full comparator

_FUNCTION = re.compile(r"void median_select<(\d+)>\(float \(&v\)\[(\d+)\]\) \{\n(.*?)^\}", re.S | re.M)
_OPERAND = r"(t|v\[\d+\])"
_ASSIGN = re.compile(r"^%s = (?:(fminf|fmaxf)\(%s, %s\)|%s)$" % (_OPERAND, _OPERAND, _OPERAND, _OPERAND))


def _operand(text):
    return TMP if text == "t" else int(text[2:-1])


def parse_header(name):
    """{n: [(op, dst, a, b)]}: every assignment of every median_select<n>, in program order.  op is "fminf",
    "fmaxf" or "mov" (b = None); operands are wire indices or TMP.  Anything else in a body is an error."""
    with open(os.path.join(CSRC, name)) as f:
        text = f.read()
    networks = {}
    for n, size, body in _FUNCTION.findall(text):
        assert n == size, name
        statements = []
        for piece in body.replace("\n", " ").split(";"):
            piece = piece.strip()
            if not piece or piece == "float t":
                continue
            m = _ASSIGN.match(piece)
            assert m, "%s, median_select<%s>: unexpected statement %r" % (name, n, piece)
            dst, op, a, b, src = m.groups()
            if op:
                statements.append((op, _operand(dst), _operand(a), _operand(b)))
            else:
                statements.append(("mov", _operand(dst), _operand(src), None))
        networks[int(n)] = statements
    return networks


def comparators(statements):
    """The statement list as the generator's (i, j, need_min, need_max) comparators.  The three shapes it emits:
    t = fminf(v[i], v[j]); v[j] = fmaxf(v[i], v[j]); v[i] = t;   v[i] = fminf(v[i], v[j]);   v[j] = fmaxf(v[i], v[j]);
    a statement outside them is returned as is, so that the comparison with the generator fails on it."""
    out, s = [], 0
    while s < len(statements):
        op, dst, a, b = statements[s]
        full = statements[s : s + 3]
        if (op == "fminf" and dst == TMP and len(full) == 3 and full[1] == ("fmaxf", b, a, b)
                and full[2] == ("mov", a, TMP, None)):
            out.append((a, b, True, True))
            s += 3
            continue
        if op == "fminf" and dst == a:
            out.append((a, b, True, False))
        elif op == "fmaxf" and dst == b:
            out.append((a, b, False, True))
        else:
            out.append(statements[s])
        s += 1
    return out


def execute(statements, wires, fmin, fmax):
    """Run a network in place on a list of per-wire arrays."""
    t = None
    for op, dst, a, b in statements:
        x = t if a == TMP else wires[a]
        if op == "mov":
            value = x
        else:
            y = t if b == TMP else wires[b]
            value = (fmin if op == "fminf" else fmax)(x, y)
        if dst == TMP:
            t = value
        else:
            wires[dst] = value


@pytest.fixture(scope="module")
def small():
    return parse_header("median_networks.cuh")


@pytest.fixture(scope="module")
def large():
    return parse_header("median_networks_large.cuh")


@pytest.fixture(scope="module")
def generator():
    spec = importlib.util.spec_from_file_location("gen_median_networks", os.path.join(ROOT, "tools", "gen_median_networks.py"))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)  # main() only runs as a script: nothing is written
    return module


def test_headers_are_what_the_generator_emits(small, large, generator):
    assert sorted(small) == list(range(1, 33))
    assert sorted(large) == [48, 64, 100, 128]
    for n, statements in list(small.items()) + list(large.items()):
        assert comparators(statements) == [tuple(c) for c in generator.median_network(n)], n


# ---- n = 1..32: every 0/1 input -------------------------------------------------------------------------
# Bit-sliced: a uint64 word holds 64 input vectors.  Wires 0..5 vary across the lanes of a word, the next
# `CHUNK_BITS` wires across the words of a chunk, the rest across chunks, so the weight of an input vector is
# popcount(lane) + popcount(word) + popcount(chunk) and the expected output word comes from a table.
CHUNK_BITS = 18
_LANES = np.arange(64, dtype=np.uint64)
_LANE_WEIGHT = np.array([bin(lane).count("1") for lane in range(64)])
_ONES = np.uint64(0xFFFFFFFFFFFFFFFF)


def _lane_word(selected):
    return np.uint64(int(np.sum(np.left_shift(np.uint64(1), _LANES[selected]), dtype=np.uint64)))


def _check_chunk(statements, n, chunk, chunk_bits):
    low = min(n, 6)
    words = 1 << chunk_bits
    index = np.arange(words, dtype=np.uint64)
    wires = []
    for w in range(n):
        if w < 6:
            wires.append(np.full(words, _lane_word((_LANES >> np.uint64(w)) & np.uint64(1) == 1), dtype=np.uint64))
        elif w < 6 + chunk_bits:
            wires.append(np.where((index >> np.uint64(w - 6)) & np.uint64(1) == 1, _ONES, np.uint64(0)))
        else:
            wires.append(np.full(words, _ONES if (chunk >> (w - 6 - chunk_bits)) & 1 else np.uint64(0), dtype=np.uint64))
    execute(statements, wires, np.bitwise_and, np.bitwise_or)
    valid = _lane_word(_LANES < (1 << low))
    high_weight = np.array([bin(i).count("1") for i in range(words)]) + bin(chunk).count("1")
    # at_least[s] = lanes whose low wires hold >= s ones, for s = 0..7
    at_least = np.array([_lane_word(_LANE_WEIGHT >= s) for s in range(8)], dtype=np.uint64)
    for rank in sorted({(n - 1) // 2, n // 2}):
        # the rank-th smallest of a 0/1 vector is 1 iff it holds at least n - rank ones
        expected = at_least[np.clip(n - rank - high_weight, 0, 7)]
        bad = np.flatnonzero((wires[rank] ^ expected) & valid)
        if bad.size:
            return "n=%d rank %d: wrong on word %d of chunk %d" % (n, rank, int(bad[0]), chunk)
    return None


def test_small_networks_select_both_middles_of_every_01_input(small):
    jobs = []
    for n in range(1, 33):
        chunk_bits = min(CHUNK_BITS, max(0, n - 6))
        jobs += [(n, chunk, chunk_bits) for chunk in range(1 << max(0, n - 6 - chunk_bits))]
    with ThreadPoolExecutor(os.cpu_count() or 4) as pool:  # NumPy releases the GIL on these arrays
        errors = [e for e in pool.map(lambda job: _check_chunk(small[job[0]], *job), jobs) if e]
    assert not errors, errors[:4]


# ---- n = 33..128 through the padded 48/64/100/128-slot networks ----------------------------------------
def _slots(n):
    """NS of the k_simmodel_large / k_simmodel_nyquist dispatch."""
    return 48 if n <= 48 else 64 if n <= 64 else 100 if n <= 100 else 128


def _vectors(n, rng):
    """(n, M) float32 columns: 0/1 vectors at the critical weights of both middle ranks, permutations of
    distinct values, and values drawn from {0, 1, 2}."""
    weights = sorted({n - r - d for r in ((n - 1) // 2, n // 2) for d in (0, 1)})
    binary = []
    for weight in weights:
        block = np.zeros((n, -(-4000 // len(weights))), dtype=np.float32)
        block[:weight] = 1
        binary.append(rng.permuted(block, axis=0))
    distinct = np.exp(rng.uniform(-8, 8, size=(n, 1))).astype(np.float32)
    assert len(np.unique(distinct)) == n
    permutations = rng.permuted(np.repeat(distinct, 3000, axis=1), axis=0)
    ties = rng.integers(0, 3, size=(n, 3000)).astype(np.float32)
    return np.concatenate(binary + [permutations, ties], axis=1)


@pytest.mark.parametrize("n", range(33, 129))
def test_large_networks_with_the_kernel_padding(large, n):
    rng = np.random.default_rng(n)
    data = _vectors(n, rng)
    count = data.shape[1]
    assert count >= 10000
    slots = _slots(n)
    lo = (slots - n) >> 1  # gather_median_large: slot s >= n holds -inf if s - n < lo, else +inf
    wires = [data[s] for s in range(n)]
    wires += [np.full(count, -np.inf if s < lo else np.inf, dtype=np.float32) for s in range(slots - n)]
    execute(large[slots], wires, np.minimum, np.maximum)
    ordered = np.sort(data, axis=0)
    assert np.array_equal(wires[slots // 2 - 1], ordered[(n - 1) // 2]), "lower middle, n=%d" % n
    if n % 2 == 0:
        assert np.array_equal(wires[slots // 2], ordered[n // 2]), "upper middle, n=%d" % n
    # the kernel's arithmetic on them (squared magnitudes in, np.median of the magnitudes out)
    root_lo = np.sqrt(wires[slots // 2 - 1].astype(np.float64))
    got = root_lo if n % 2 else 0.5 * (root_lo + np.sqrt(wires[slots // 2].astype(np.float64)))
    assert np.array_equal(got, np.median(np.sqrt(data.astype(np.float64)), axis=0)), n
