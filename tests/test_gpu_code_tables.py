"""The device codec on code tables other than HPACK's, through every encode and decode route.

The library takes any prefix code of codes up to 32 bits, and its fast kernels size and choose themselves from
properties of the table: the shortest code (batch decoder rows and strings per tile, whether the fused stream kernel
runs, the one-kernel HPACK literal route), the longest code (fast encoders up to 31 bits, sub-table depth), two-symbol
root entries, the LUT size (fast decoders up to 8192 entries, then the generic decoder with the LUT split between
shared and global memory) and codeless symbols (generic encode). Each table below is built from a list of code
lengths (canonical codes, `oracle/table_builder_oracle.py`) or from explicit patterns, never with the product's
builder, and lands on one of those edges.

CPU part (-m "not gpu"): every table is a prefix code with the intended shortest and longest code, Kraft sum and LUT
size, and a pure-Python bit-string codec agrees with the oracle on every table (the oracle had only been pinned on the
two shipped tables).
GPU part: every route, forced or chosen by the table, against the oracle, every output array compared."""
import ctypes as C
import functools
import importlib.util
import os
from fractions import Fraction

import numpy as np
import pytest

import refcodec
from refcodec import OK, SHORT_BUFFER, UNKNOWN_SYMBOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "oracle", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


tbo = _load("table_builder_oracle")
lit = _load("hpack_literals_oracle")

LUT_ROOT_BITS, LUT_SUB_BITS, LUT_MAX_FAST = 12, 8, 8192  # the device LUT layout (csrc/huffman_batch.cu)


# ---------------------------------------------------------------------------------------------------------------
# the tables
# ---------------------------------------------------------------------------------------------------------------

def _complete_lengths(shortest, longest, n=256):
    """Code lengths of a complete code of n symbols: one code of `shortest` bits, a spine of codes down to two of
    `longest` bits, and the rest split evenly (the shallowest code split first) until there are n codes."""
    fixed = [shortest, longest, longest]
    pool = [shortest] * (2 ** shortest - 2) + list(range(shortest + 1, longest))
    while len(fixed) + len(pool) < n:
        pool.sort()
        length = pool.pop(0)
        pool += [length + 1, length + 1]
    return fixed + pool


def _canonical(lengths, seed):
    """Deals `lengths` to the symbols in a seeded order (the rest get no code); canonical patterns."""
    order = np.random.default_rng(seed).permutation(256)
    num_bits = np.zeros(256, dtype=np.uint8)
    for sym, length in zip(order, lengths):
        num_bits[sym] = length
    codes, _ = tbo.canonical([int(x) for x in num_bits])
    patterns = np.zeros(256, dtype=np.uint32)
    for sym, (pattern, _) in codes.items():
        patterns[sym] = pattern
    return patterns, num_bits


def _lut_family(with_17_bit_code):
    """256 codes of 16 bits under 256 distinct 12-bit prefixes: every prefix owns a 16-entry sub-table (4096 + 256 x 16
    = 8192 LUT entries). With the 17-bit code, the last prefix owns a 32-entry sub-table instead (8208)."""
    order = np.random.default_rng(16).permutation(256)
    patterns = np.zeros(256, dtype=np.uint32)
    num_bits = np.zeros(256, dtype=np.uint8)
    for i, sym in enumerate(order):
        prefix = 16 * i + (5 * i) % 16
        if with_17_bit_code and i == 255:
            patterns[sym], num_bits[sym] = (prefix << 5) | 0b10110, 17
        else:
            patterns[sym], num_bits[sym] = (prefix << 4) | ((7 * i) & 15), 16
    return patterns, num_bits


def _flat8():
    patterns = np.random.default_rng(8).permutation(256).astype(np.uint32)  # encode is a byte map
    return patterns, np.full(256, 8, dtype=np.uint8)


def _few(codes):
    patterns = np.zeros(256, dtype=np.uint32)
    num_bits = np.zeros(256, dtype=np.uint8)
    for sym, (pattern, length) in codes.items():
        patterns[sym], num_bits[sym] = pattern, length
    return patterns, num_bits


def _sparse():
    rng = np.random.default_rng(40)
    syms = rng.choice(256, size=40, replace=False)
    lengths = np.zeros(256, dtype=np.int64)
    lengths[syms] = [3] * 2 + [6] * 14 + [8] * 24
    codes, _ = tbo.canonical([int(x) for x in lengths])
    return _few(codes)


_MAX31 = [8] * 223 + [10] * 4 + list(range(4, 31)) + [31, 31]
_MAX32 = [8] * 223 + [10] * 4 + list(range(4, 30)) + [31, 32, 32]

# name: (builder, shortest, longest, Kraft sum, LUT entries or None for "at most 8192")
SPECS = {
    "flat8": (_flat8, 8, 8, Fraction(1), 4096),
    "min1": (lambda: _canonical(_complete_lengths(1, 14), 1), 1, 14, Fraction(1), None),
    "min2": (lambda: _canonical(_complete_lengths(2, 13), 2), 2, 13, Fraction(1), None),
    "min3": (lambda: _canonical(_complete_lengths(3, 16), 3), 3, 16, Fraction(1), None),
    "min4": (lambda: _canonical(_complete_lengths(4, 13), 4), 4, 13, Fraction(1), None),
    "min6": (lambda: _canonical(_complete_lengths(6, 13), 6), 6, 13, Fraction(1), None),
    "min7": (lambda: _canonical(_complete_lengths(7, 13), 7), 7, 13, Fraction(1), None),
    "max12": (lambda: _canonical(_complete_lengths(5, 12), 12), 5, 12, Fraction(1), 4096),
    "max13": (lambda: _canonical(_complete_lengths(5, 13), 13), 5, 13, Fraction(1), None),
    "max20": (lambda: _canonical(_complete_lengths(5, 20), 20), 5, 20, Fraction(1), None),
    "max21": (lambda: _canonical(_complete_lengths(5, 21), 21), 5, 21, Fraction(1), None),
    "max31": (lambda: _canonical(_MAX31, 31), 4, 31, Fraction(1), 4616),
    "max32": (lambda: _canonical(_MAX32, 32), 4, 32, 1 - Fraction(1, 1 << 30), 4624),
    "lut8192": (lambda: _lut_family(False), 16, 16, Fraction(1, 256), 8192),
    "lut8208": (lambda: _lut_family(True), 16, 17, Fraction(255, 65536) + Fraction(1, 1 << 17), 8208),
    "one_symbol": (lambda: _few({0x61: (0, 1)}), 1, 1, Fraction(1, 2), 4096),
    "two_symbols": (lambda: _few({0x61: (0, 1), 0x62: (1, 1)}), 1, 1, Fraction(1), 4096),
    "sparse": (_sparse, 3, 8, Fraction(2, 8) + Fraction(14, 64) + Fraction(24, 256), 4096),
}
NAMES = list(SPECS)
SUB_TABLE_DEPTH = {"max12": 0, "max13": 1, "max20": 1, "max21": 2}


@functools.lru_cache(maxsize=None)
def table_arrays(name):
    patterns, num_bits = SPECS[name][0]()
    patterns.setflags(write=False)
    num_bits.setflags(write=False)
    return patterns, num_bits


# ---- a second reading of the code, in plain Python ----------------------------------------------------------------

def _trie(patterns, num_bits):
    root = {}
    for sym in range(256):
        length = int(num_bits[sym])
        if not length:
            continue
        node = root
        bits = format(int(patterns[sym]), "0%db" % length)
        for b in bits[:-1]:
            node = node.setdefault(b, {})
            assert isinstance(node, dict), "a code is a prefix of another"
        assert bits[-1] not in node, "a code is a prefix of another"
        node[bits[-1]] = sym
    return root


def _height(node):
    return 0 if not isinstance(node, dict) else 1 + max(_height(c) for c in node.values())


def _below(node, depth):
    """The inner nodes exactly `depth` levels below `node`."""
    if depth == 0:
        yield node
        return
    for child in node.values():
        if isinstance(child, dict):
            yield from _below(child, depth - 1)


def lut_layout(patterns, num_bits):
    """(entries, sub-table depth) of the two-level LUT: a 2^12 root, and under every inner node at the bottom of a
    table a sub-table 2^min(height, 8) wide."""
    def table(node, width):
        entries, depth = 1 << width, 0
        for inner in _below(node, width):
            e, d = table(inner, min(_height(inner), LUT_SUB_BITS))
            entries, depth = entries + e, max(depth, d + 1)
        return entries, depth
    return table(_trie(patterns, num_bits), LUT_ROOT_BITS)


def py_encode(patterns, num_bits, eos, data):
    """(status, consumed, bytes): the codes one after another; the last byte filled with the low bits of the padding
    byte; a symbol without a code stops the string after the whole bytes written so far."""
    bits = []
    for i, sym in enumerate(bytes(data)):
        length = int(num_bits[sym])
        if not length:
            whole = "".join(bits)
            return UNKNOWN_SYMBOL, i + 1, bytes(int(whole[k:k + 8], 2) for k in range(0, len(whole) // 8 * 8, 8))
        bits.append(format(int(patterns[sym]), "0%db" % length))
    whole = "".join(bits)
    free = -len(whole) % 8
    if free:
        whole += format(eos & ((1 << free) - 1), "0%db" % free)
    return OK, len(data), bytes(int(whole[k:k + 8], 2) for k in range(0, len(whole), 8))


def py_decode(codes, data):
    """(status, symbols): the longest-prefix walk over the bits, with zeros after the end; no code in the next 32 bits
    is an unknown symbol when 32 bits or more are left, and the end otherwise; a code running past the end is the end."""
    bits = "".join(format(b, "08b") for b in bytes(data))
    longest = max(len(c) for c in codes)
    out, pos = bytearray(), 0
    while pos < len(bits):
        window = (bits[pos:pos + 32] + "0" * 32)[:32]
        hit = next(((codes[window[:k]], k) for k in range(1, longest + 1) if window[:k] in codes), None)
        if hit is None:
            return (UNKNOWN_SYMBOL if len(bits) - pos >= 32 else OK), bytes(out)
        if hit[1] > len(bits) - pos:
            break
        out.append(hit[0])
        pos += hit[1]
    return OK, bytes(out)


def code_strings(patterns, num_bits):
    return {format(int(patterns[s]), "0%db" % int(num_bits[s])): s for s in range(256) if num_bits[s]}


# ---- seeded inputs ------------------------------------------------------------------------------------------------

def coded_symbols(name):
    return np.flatnonzero(table_arrays(name)[1]).astype(np.uint8)


def sampler(name, coded_only):
    """Zipf over the symbols ranked by code length (the short codes most often); coded_only keeps symbols without a
    code out."""
    s = refcodec.zipf_symbol_sampler(table_arrays(name)[1])
    if coded_only:
        coded = coded_symbols(name)
        s = np.where(np.isin(s, coded), s, coded[0]).astype(np.uint8)
    return s


def symbols(rng, name, size, kind):
    if kind == "zipf":
        return np.ascontiguousarray(sampler(name, True)[rng.integers(0, 65536, size=size)])
    if kind == "zipf_all":
        return np.ascontiguousarray(sampler(name, False)[rng.integers(0, 65536, size=size)])
    if kind == "uniform":
        return np.ascontiguousarray(rng.choice(coded_symbols(name), size=size))
    if kind == "bytes":
        return rng.integers(0, 256, size=size, dtype=np.uint8)
    if kind == "longest":  # the (up to) 8 symbols with the longest codes
        nb = table_arrays(name)[1]
        longest = np.argsort(-nb.astype(np.int64), kind="stable")[:8]
        return np.ascontiguousarray(rng.choice(longest[nb[longest] > 0], size=size).astype(np.uint8))
    raise KeyError(kind)


def offsets(lens):
    offs = np.zeros(len(lens) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(np.asarray(lens, dtype=np.int64))
    return offs


def batch(rng, name, lens, kind):
    offs = offsets(lens)
    return symbols(rng, name, int(offs[-1]), kind), offs


def with_runs(rng, payload, share=0.5):
    """Overwrites about `share` of the bytes with runs of 0x00 and of 0xFF, 1..40 bytes long."""
    payload = payload.copy()
    pos = 0
    while pos < len(payload):
        pos += int(rng.integers(0, 40))
        run = int(rng.integers(1, 41))
        if rng.random() < share:
            payload[pos:pos + run] = 0xFF if rng.random() < 0.5 else 0x00
        pos += run
    return payload


def flip_bits(rng, payload, every=60):
    payload = payload.copy()
    if len(payload):
        where = rng.integers(0, len(payload), size=max(1, len(payload) // every))
        payload[where] ^= (1 << rng.integers(0, 8, size=len(where))).astype(np.uint8)
    return payload


# ---------------------------------------------------------------------------------------------------------------
# CPU: the tables are what they claim, and the oracle reads every one of them like the plain restatement above
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", NAMES)
def test_table_shape(oracle, name):
    _, shortest, longest, kraft, lut = SPECS[name]
    patterns, num_bits = table_arrays(name)
    oracle.table(patterns, num_bits)  # raises unless prefix-free
    lengths = [int(x) for x in num_bits if x]
    assert (min(lengths), max(lengths)) == (shortest, longest)
    assert sum(Fraction(1, 1 << x) for x in lengths) == kraft
    assert all(int(patterns[s]) < (1 << int(num_bits[s])) for s in range(256) if num_bits[s])
    entries, depth = lut_layout(patterns, num_bits)
    if lut is None:
        assert entries <= LUT_MAX_FAST
    else:
        assert entries == lut
    if name in SUB_TABLE_DEPTH:
        assert depth == SUB_TABLE_DEPTH[name]
    if name == "flat8":
        assert sorted(patterns.tolist()) == list(range(256))


def test_table_edges_are_where_the_dispatch_turns():
    """What each table is for: the fused stream kernel's row check (csrc/huffman_batch.cu, decode_stream_fast) is on
    from a shortest code of 5 bits; no root entry can hold two symbols from 7."""
    def fused(min_len):
        stage = ((257 * 33 + 1) * 4 + 15) & ~15
        row_words = (((1024 + 31) // min_len + 4 + 3) // 4) | 1
        return 256 * row_words * 4 + 16 <= 2 * stage - row_words * 4 - 32
    assert [fused(m) for m in range(1, 9)] == [False] * 4 + [True] * 4
    assert {SPECS[n][1] for n in ("min1", "min2", "min3", "min4")} == {1, 2, 3, 4}
    assert {SPECS[n][1] for n in ("min6", "min7")} == {6, 7}
    assert 2 * SPECS["min7"][1] > LUT_ROOT_BITS >= 2 * SPECS["min6"][1]


@pytest.mark.parametrize("name", NAMES)
def test_python_codec_agrees_with_the_oracle(oracle, name):
    rng = np.random.default_rng(sum(map(ord, name)))
    patterns, num_bits = table_arrays(name)
    table = oracle.table(patterns, num_bits)
    codes = code_strings(patterns, num_bits)
    n = 300
    for kind in ("zipf", "zipf_all", "bytes"):
        data, offs = batch(rng, name, rng.integers(0, 60, size=n), kind)
        for eos in (0xFF, 0x00, 0xA5):
            want = oracle.encode_batch(table, eos, data, offs, 4 * len(data) + 64)
            for i in range(n):
                status, consumed, out = py_encode(patterns, num_bits, eos, data[int(offs[i]):int(offs[i + 1])])
                a = int(want["out_offsets"][i])
                assert (status, consumed) == (int(want["status"][i]), int(want["consumed"][i])), (kind, eos, i)
                assert out == bytes(want["out"][a:a + int(want["out_lens"][i])]), (kind, eos, i)
        if kind == "zipf_all":
            continue
        # decode: the clean encodings, then arbitrary bytes with runs of zeros and ones
        enc = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
        stream = enc["out"][:int(enc["out_offsets"][-1])]
        for payload, poffs in ((stream, enc["out_offsets"]), (with_runs(rng, stream), enc["out_offsets"])):
            want = oracle.decode_batch(table, payload, poffs, 8 * len(payload) + 64)
            for i in range(n):
                status, out = py_decode(codes, payload[int(poffs[i]):int(poffs[i + 1])])
                a = int(want["out_offsets"][i])
                assert status == int(want["status"][i]), (kind, i)
                assert out == bytes(want["out"][a:a + int(want["out_lens"][i])]), (kind, i)
                if payload is stream and kind == "zipf":  # (padding bits that form a code decode as symbols)
                    assert status == OK and out.startswith(bytes(data[int(offs[i]):int(offs[i + 1])])), i


def test_flat8_encode_is_a_byte_map(oracle):
    patterns, num_bits = table_arrays("flat8")
    data = np.random.default_rng(3).integers(0, 256, size=5000, dtype=np.uint8)
    want = oracle.encode_batch(oracle.table(patterns, num_bits), 0xA5, data, [0, len(data)], len(data) + 8)
    assert bytes(want["out"][:len(data)]) == data.tobytes().translate(bytes(patterns.astype(np.uint8)))


def test_literal_oracle_decodes_codes_shorter_than_two_bits(oracle):
    """A literal of 1-bit codes decodes to eight symbols per octet (the literal oracle once sized its output for two)."""
    patterns, num_bits = table_arrays("min1")
    lo = lit.LiteralOracle(oracle, oracle.table(patterns, num_bits))
    short = int(np.flatnonzero(num_bits == 1)[0])
    text = bytes([short]) * 400
    framed = lo.encode(text, lit.ALWAYS)
    assert framed[:1] == bytes([0x80 | 50]) and len(framed) == 1 + 50
    assert lo.decode(framed) == (lit.OK, text)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------

SWITCHES = {
    "default": (),
    "generic": ("AWS_HUFFMAN_BATCH_FORCE_GENERIC",),
    "no_strings": ("AWS_HUFFMAN_BATCH_NO_STRINGS",),
    "no_slots": ("AWS_HUFFMAN_BATCH_NO_SLOTS",),
    "tiled": ("AWS_HUFFMAN_BATCH_NO_STRINGS", "AWS_HUFFMAN_BATCH_NO_SLOTS"),
    "no_fused": ("AWS_HUFFMAN_BATCH_NO_FUSED_STREAM",),
}
ALL_SWITCHES = sorted({v for vs in SWITCHES.values() for v in vs})


@pytest.fixture(scope="module")
def contexts(pkg):
    """contexts(name, route, eos): a context built from the table's codes (aws_huffman_batch_ctx_new_from_code_table)
    with the route's switches set while it is created, and only those."""
    made = {}

    def get(name, route="default", eos=0xFF):
        key = (name, route, eos)
        if key not in made:
            patterns, num_bits = table_arrays(name)
            codes = (pkg.capi.aws_huffman_code * 256)()
            for s in range(256):
                codes[s].pattern, codes[s].num_bits = int(patterns[s]), int(num_bits[s])
            with pytest.MonkeyPatch.context() as mp:
                for var in ALL_SWITCHES:
                    mp.delenv(var, raising=False)
                for var in SWITCHES[route]:
                    mp.setenv(var, "1")
                made[key] = pkg.BatchContext(None, eos_padding=eos, device=0, code_table=codes)
        return made[key]

    yield get
    for ctx in made.values():
        ctx.close()


@pytest.fixture(scope="module")
def oracle_table(oracle):
    made = {}

    def get(name):
        if name not in made:
            made[name] = oracle.table(*table_arrays(name))
        return made[name]
    return get


def assert_same(got, want, what, whole_out=False):
    for key in want:
        if key == "out":
            continue
        g, w = np.asarray(got[key]), np.asarray(want[key])
        bad = np.flatnonzero(g != w)
        assert not len(bad), "%s: %s differs first at %s (got %s, want %s)" % (what, key, bad[:5], g[bad[:3]], w[bad[:3]])
    end = len(want["out"]) if whole_out else int(want["out_offsets"][-1])
    bad = np.flatnonzero(got["out"][:end] != want["out"][:end])
    assert not len(bad), "%s: out differs first at byte %s" % (what, bad[:5])


def slots_around(rng, need, lo, hi):
    caps = np.maximum(0, need.astype(np.int64) + rng.integers(lo, hi, size=len(need))).astype(np.uint64)
    slots = np.zeros(len(caps), dtype=np.uint64)
    slots[1:] = np.cumsum(caps)[:-1]
    return slots, caps, int(caps.sum()) + 1


ENCODE_ROUTES = [("default", 0xFF), ("default", 0x00), ("default", 0xA5), ("generic", 0xA5), ("no_strings", 0x00),
                 ("no_slots", 0xFF), ("tiled", 0xA5)]


def encode_inputs(rng, name):
    yield "short_zipf", batch(rng, name, rng.integers(0, 301, size=2500), "zipf_all")
    yield "short_bytes", batch(rng, name, rng.integers(0, 301, size=1200), "bytes")
    yield "avg_over_2k", batch(rng, name, rng.integers(2048, 6000, size=40), "zipf")
    # items starting on, just before and just after the 8 KiB tiles and 32-symbol thread ranges
    yield "tile_edges", batch(rng, name, [8192, 0, 0, 1, 8191, 31, 1, 32, 0, 33, 8192 * 2 - 97, 97, 5, 0, 8192, 3], "zipf")
    for n in (1, 8191, 8192, 8193, 8192 * 2 + 31, 8192 * 2 + 32, 8192 * 2 + 33):
        yield "single_%d" % n, batch(rng, name, [n], "zipf")
    # short strings, and three whose encoding passes 8 KiB when the longest codes are over 21 bits (the string
    # encoder leaves those to the tiled kernel)
    lens = rng.integers(0, 301, size=600)
    data, offs = batch(rng, name, lens, "zipf")
    long_items = [symbols(rng, name, 3000, "longest") for _ in range(3)]
    at = [100, 101, 400]
    pieces, k = [], 0
    for i in range(len(lens)):
        pieces.append(data[int(offs[i]):int(offs[i + 1])])
        if i in at:
            pieces.append(long_items[k])
            k += 1
    yield "long_codes_past_8k", (np.ascontiguousarray(np.concatenate(pieces)), offsets([len(p) for p in pieces]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_encode_routes_match_the_oracle(contexts, oracle, oracle_table, name):
    rng = np.random.default_rng(0xE0 + NAMES.index(name))
    table = oracle_table(name)
    for label, (data, offs) in encode_inputs(rng, name):
        cap = 4 * len(data) + 64
        wants = {}
        for route, eos in ENCODE_ROUTES:
            if eos not in wants:
                wants[eos] = oracle.encode_batch(table, eos, data, offs, cap)
            got = contexts(name, route, eos).encode(data, offs, cap)
            assert_same(got, wants[eos], "%s %s eos=%#x" % (label, route, eos))
        ctx = contexts(name)
        assert np.array_equal(ctx.encoded_lengths(data, offs),
                              [oracle.encoded_length(table, data[int(offs[i]):int(offs[i + 1])])
                               for i in range(len(offs) - 1)]), label
    # slotted layout: capacities scattered around the need, bytes around the slots untouched
    data, offs = batch(rng, name, rng.integers(0, 301, size=2500), "zipf_all")
    need = oracle.encode_batch(table, 0xA5, data, offs, 4 * len(data) + 64)["out_lens"]
    slots, caps, total = slots_around(rng, need, -8, 3)
    sentinel = np.full(total, 0x5A, dtype=np.uint8)
    want = oracle.encode_batch(table, 0xA5, data, offs, total, out_offsets=slots, out_caps=caps, out=sentinel.copy())
    for route in ("default", "generic"):
        got = contexts(name, route, 0xA5).encode(data, offs, total, out_offsets=slots, out_caps=caps, out=sentinel.copy())
        assert_same(got, want, "slotted %s" % route, whole_out=True)
    assert (want["status"] == SHORT_BUFFER).any()


def decode_batches(rng, name, oracle, table):
    """(label, payload, offsets) of many-item batches."""
    for kind in ("zipf", "uniform"):
        data, offs = batch(rng, name, rng.integers(0, 301, size=2500), kind)
        enc = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
        stream = enc["out"][:int(enc["out_offsets"][-1])]
        yield "clean_" + kind, stream, enc["out_offsets"]
        yield "flipped_" + kind, flip_bits(rng, stream), enc["out_offsets"]
    lens = rng.integers(0, 121, size=3000)
    yield "bytes_short", with_runs(rng, rng.integers(0, 256, size=int(lens.sum()), dtype=np.uint8)), offsets(lens)
    yield "zeros_short", np.zeros(int(lens.sum()), dtype=np.uint8), offsets(lens)
    # 500..3000 B strings: with 1- and 2-bit codes a tile's rows overflow and it takes the two-pass route
    lens = rng.integers(500, 3001, size=60)
    yield "zeros_long", np.zeros(int(lens.sum()), dtype=np.uint8), offsets(lens)
    yield "bytes_long", with_runs(rng, rng.integers(0, 256, size=int(lens.sum()), dtype=np.uint8)), offsets(lens)
    lens = rng.integers(0, 300, size=2000)
    lens[[7, 900, 901, 1500]] = [3000, 2600, 40000, 70000]
    yield "zeros_mixed", with_runs(rng, np.zeros(int(lens.sum()), dtype=np.uint8), 0.05), offsets(lens)


def clean_stream(rng, name, oracle, table, encoded_bytes):
    nb = table_arrays(name)[1].astype(np.float64)
    probe = symbols(rng, name, 65536, "zipf")
    n = int(encoded_bytes * 8 / nb[probe].mean()) + 1
    data = symbols(rng, name, n, "zipf")
    enc = oracle.encode_batch(table, 0xFF, data, [0, n], 4 * n + 64)
    return enc["out"][:int(enc["out_offsets"][-1])].copy()


def decode_streams(rng, name, oracle, table):
    """(label, payload) of single items long enough for the stream kernels (64 KiB and up)."""
    stream = clean_stream(rng, name, oracle, table, 90_000)
    yield "stream_clean", stream
    yield "stream_flipped", flip_bits(rng, stream, every=20_000)
    yield "stream_zeros", np.zeros(72_000, dtype=np.uint8)
    yield "stream_bytes", with_runs(rng, rng.integers(0, 256, size=80_000, dtype=np.uint8))
    base = (len(stream) // 128 - 3) * 128  # a multiple of the 128-byte chunk
    for cut in range(base - 1, base + 6):
        yield "stream_cut_%d" % (cut - base), stream[:cut].copy()


BIG_STREAMS = ("min1", "min3", "min6", "max21", "max31", "lut8192", "lut8208")


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_decode_routes_match_the_oracle(contexts, oracle, oracle_table, name):
    rng = np.random.default_rng(0xD0 + NAMES.index(name))
    table = oracle_table(name)
    for label, payload, offs in decode_batches(rng, name, oracle, table):
        cap = 8 * len(payload) + 64
        want = oracle.decode_batch(table, payload, offs, cap)
        for route in ("default", "generic"):
            assert_same(contexts(name, route).decode(payload, offs, cap), want, "%s %s" % (label, route))
        if label == "clean_zipf":
            assert (want["status"] == OK).all()
            slots, caps, total = slots_around(rng, want["out_lens"], -6, 2)
            want_s = oracle.decode_batch(table, payload, offs, total, out_offsets=slots, out_caps=caps)
            for route in ("default", "generic"):
                got = contexts(name, route).decode(payload, offs, total, out_offsets=slots, out_caps=caps)
                assert_same(got, want_s, "slotted %s" % route, whole_out=True)
    for label, payload in decode_streams(rng, name, oracle, table):
        offs = np.array([0, len(payload)], dtype=np.uint64)
        cap = 8 * len(payload) + 64
        want = oracle.decode_batch(table, payload, offs, cap)
        for route in ("default", "no_fused", "generic"):
            assert_same(contexts(name, route).decode(payload, offs, cap), want, "%s %s" % (label, route))
    if name in BIG_STREAMS:
        payload = clean_stream(rng, name, oracle, table, 3_000_000)
        offs = np.array([0, len(payload)], dtype=np.uint64)
        want = oracle.decode_batch(table, payload, offs, 8 * len(payload) + 64)
        for route in ("default", "no_fused"):
            assert_same(contexts(name, route).decode(payload, offs, 8 * len(payload) + 64), want, "3 MB %s" % route)


def launches(ctx, call):
    before = ctx.launch_count
    call(ctx)
    return ctx.launch_count - before


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_stream_route_follows_the_shortest_code(contexts, oracle, oracle_table, name):
    """On one stream the fused kernel and its verify pass run (two launches more than the multi-kernel twin) exactly
    when the shortest code has 5 bits or more and the LUT fits shared memory."""
    rng = np.random.default_rng(0x5E + NAMES.index(name))
    table = oracle_table(name)
    payload = clean_stream(rng, name, oracle, table, 90_000)
    offs = np.array([0, len(payload)], dtype=np.uint64)
    cap = 8 * len(payload) + 64
    want = oracle.decode_batch(table, payload, offs, cap)
    counts = {}
    for route in ("default", "no_fused"):
        got = {}
        counts[route] = launches(contexts(name, route), lambda c: got.update(c.decode(payload, offs, cap)))
        assert_same(got, want, route)
    fused = SPECS[name][1] >= 5 and lut_layout(*table_arrays(name))[0] <= LUT_MAX_FAST
    assert counts["default"] - counts["no_fused"] == (2 if fused else 0), counts


@pytest.mark.gpu
def test_batch_decode_route_follows_the_lut_size(contexts, oracle, oracle_table):
    """8192 LUT entries decode in the one fast kernel; 8208 take the generic decoder, whose LUT does not fit its
    shared memory (its first 8192 entries are there, the rest is read from global memory)."""
    counts = {}
    for name in ("lut8192", "lut8208"):
        rng = np.random.default_rng(82)
        table = oracle_table(name)
        data, offs = batch(rng, name, rng.integers(0, 200, size=3000), "uniform")
        enc = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
        payload = with_runs(rng, enc["out"][:int(enc["out_offsets"][-1])], 0.1)
        cap = 8 * len(payload) + 64
        want = oracle.decode_batch(table, payload, enc["out_offsets"], cap)
        for route in ("default", "generic"):
            got = {}
            counts[name, route] = launches(contexts(name, route),
                                           lambda c: got.update(c.decode(payload, enc["out_offsets"], cap)))
            assert_same(got, want, "%s %s" % (name, route))
    assert counts["lut8192", "default"] == 1 and counts["lut8192", "generic"] > 1, counts
    assert counts["lut8208", "default"] == counts["lut8208", "generic"], counts


@pytest.mark.gpu
def test_encode_route_follows_the_longest_code(contexts, oracle, oracle_table):
    """Codes of 31 bits still take the fast encoders (the string encoder: prep, bits, scan, pack, the gated tiled redo
    and the per-item arrays); one 32-bit code sends the batch to the generic encoder."""
    counts = {}
    for name in ("max31", "max32"):
        rng = np.random.default_rng(31)
        table = oracle_table(name)
        data, offs = batch(rng, name, rng.integers(0, 301, size=3000), "longest")
        want = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
        for route in ("default", "generic"):
            got = {}
            counts[name, route] = launches(contexts(name, route),
                                           lambda c: got.update(c.encode(data, offs, 4 * len(data) + 64)))
            assert_same(got, want, "%s %s" % (name, route))
    assert counts["max31", "default"] != counts["max31", "generic"], counts
    assert counts["max32", "default"] == counts["max32", "generic"], counts


# ---- HPACK string literals ----------------------------------------------------------------------------------------

LITERAL_TABLES = ("min1", "min4", "flat8", "lut8192", "lut8208")


def literal_strings(rng, name, n):
    lens = rng.integers(0, 201, size=n)
    lens[rng.choice(n, size=6, replace=False)] = [126, 127, 128, 300, 5000, 0]
    data, offs = batch(rng, name, lens, "zipf")
    for i in rng.choice(n, size=n // 10, replace=False):
        a, b = int(offs[i]), int(offs[i + 1])
        data[a:b] = symbols(rng, name, b - a, "uniform")
    return data, offs


def damaged(rng, framed, f_offs):
    """Every 7th literal damaged: cut short, an octet left over, padding bits cleared, a whole octet of padding,
    nothing at all, an unfinished length, a length beyond 64 bits."""
    items = [bytearray(framed[int(f_offs[i]):int(f_offs[i + 1])]) for i in range(len(f_offs) - 1)]
    for k, i in enumerate(range(3, len(items), 7)):
        it, kind = items[i], k % 7
        if kind == 0 and len(it) > 1:
            del it[-1]
        elif kind == 1:
            it.append(0x00)
        elif kind == 2 and len(it) > 1 and it[0] & 0x80:
            it[-1] &= 0xF0
        elif kind == 3 and it[0] & 0x80 and (it[0] & 0x7F) < 126:
            it[0] += 1
            it.append(0xFF)
        elif kind == 4:
            items[i] = bytearray()
        elif kind == 5:
            items[i] = bytearray([0x7F, 0x80, 0x80])
        elif kind == 6:
            items[i] = bytearray([0xFF] + [0xFF] * 10 + [0x01])
    offs = offsets([len(x) for x in items])
    return np.frombuffer(b"".join(bytes(x) for x in items), dtype=np.uint8), offs


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["chosen", "passes"])
@pytest.mark.parametrize("name", LITERAL_TABLES)
def test_hpack_literals_match_the_oracle(contexts, oracle, oracle_table, monkeypatch, name, route):
    """chosen: the route the table picks (the one-kernel decoder up to a shortest code of 8 bits and 8192 LUT entries,
    the passes around the codec above that); passes: AWS_HUFFMAN_HPACK_PASSES set."""
    monkeypatch.delenv("AWS_HUFFMAN_BATCH_FORCE_GENERIC", raising=False)
    if route == "passes":
        monkeypatch.setenv("AWS_HUFFMAN_HPACK_PASSES", "1")
    else:
        monkeypatch.delenv("AWS_HUFFMAN_HPACK_PASSES", raising=False)
    rng = np.random.default_rng(0x11 + LITERAL_TABLES.index(name))
    lo = lit.LiteralOracle(oracle, oracle_table(name))
    ctx = contexts(name)
    data, offs = literal_strings(rng, name, 1500)
    framed = {}
    for mode in (lit.SMALLEST, lit.NEVER, lit.ALWAYS):
        want, want_offs = lo.encode_batch(data, offs, mode)
        got = ctx.hpack_encode_strings(data, offs, out_capacity=len(want) + 64, mode=mode)
        assert np.array_equal(got["out_offsets"], want_offs), "mode %d offsets" % mode
        assert np.array_equal(got["out"][:len(want)], want), "mode %d bytes" % mode
        framed[mode] = (want, want_offs)
    for mode in (lit.SMALLEST, lit.ALWAYS):
        for label, (f, f_offs) in (("clean", framed[mode]), ("damaged", damaged(rng, *framed[mode]))):
            want, want_offs, want_status = lo.decode_batch(f, f_offs)
            got = ctx.hpack_decode_strings(f, f_offs, out_capacity=2 * len(data) + 4096)
            what = "mode %d %s" % (mode, label)
            assert np.array_equal(got["status"], want_status), (what, np.flatnonzero(got["status"] != want_status)[:10])
            assert np.array_equal(got["out_offsets"], want_offs), what
            assert np.array_equal(got["out"][:len(want)], want), what
            if label == "clean":
                assert (want_status == lit.OK).all() and np.array_equal(want, data), what


# ---- streaming continuation (aws_huffman_{en,de}code_batch_resume) -------------------------------------------------

def _csr(chunks):
    offs = offsets([len(c) for c in chunks])
    data = np.concatenate([np.asarray(c, dtype=np.uint8) for c in chunks]) if int(offs[-1]) else np.zeros(0, np.uint8)
    return data, offs


def resume_texts(rng, name, n):
    texts = []
    for i in range(n):
        kind = ("zipf", "uniform", "longest")[i % 3]
        texts.append(symbols(rng, name, int(rng.integers(0, 60)), kind))
    return texts


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["min1", "max32"])
def test_resume_encode_with_output_in_pieces(contexts, oracle, oracle_table, name):
    """Each string is encoded into 1..5 octets a call; 31- and 32-bit codes stay pending across 1-octet outputs."""
    rng = np.random.default_rng(0x7E + len(name))
    table = oracle_table(name)
    ctx = contexts(name, "default", 0xA5)
    n = 150
    texts = resume_texts(rng, name, n)
    encoders = [oracle.new_encoder(table, 0xA5) for _ in range(n)]
    pos = np.zeros(n, dtype=np.int64)
    done = np.zeros(n, dtype=bool)
    state = (np.zeros(n, np.uint32), np.zeros(n, np.uint8))
    rounds = pending = 0
    while not done.all():
        rounds += 1
        assert rounds < 1000
        live = np.flatnonzero(~done)
        chunks = [texts[i][pos[i]:] for i in live]
        data, in_off = _csr(chunks)
        caps = rng.integers(1, 6, size=len(live)).astype(np.uint64)
        slots = np.zeros(len(live), dtype=np.uint64)
        slots[1:] = np.cumsum(caps)[:-1]
        got = ctx.encode(data, in_off, out_capacity=int(caps.sum()) + 8, out_offsets=slots, out_caps=caps,
                         state=(state[0][live], state[1][live]))
        for j, i in enumerate(live):
            cap, a = int(caps[j]), int(slots[j])
            out = np.zeros(cap, dtype=np.uint8)
            rc, used, olen = oracle.encode_call(encoders[i], chunks[j], out, 0, cap)
            what = "string %d round %d" % (i, rounds)
            assert (int(got["status"][j]), int(got["consumed"][j]), int(got["out_lens"][j])) == (rc, used, olen), what
            assert np.array_equal(got["out"][a:a + olen], out[:olen]), what
            bits = encoders[i].overflow_bits.num_bits
            assert int(got["overflow_num_bits"][j]) == bits, what
            if bits:
                assert int(got["overflow_pattern"][j]) == encoders[i].overflow_bits.pattern, what
                pending += bits >= 24
            pos[i] += used
            state[0][i], state[1][i] = got["overflow_pattern"][j], got["overflow_num_bits"][j]
            assert rc in (OK, SHORT_BUFFER)
            done[i] = rc == OK
    if name == "max32":
        assert pending > 0, "no long code was left pending"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["min1", "max32"])
def test_resume_decode_fed_in_chunks(contexts, oracle, oracle_table, name):
    """Each encoding reaches its decoder 1..7 octets at a time, into output buffers of 1..40 octets."""
    rng = np.random.default_rng(0x7D + len(name))
    table = oracle_table(name)
    ctx = contexts(name)
    n = 150
    texts = resume_texts(rng, name, n)
    data, offs = _csr(texts)
    enc = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
    streams = [enc["out"][int(enc["out_offsets"][i]):int(enc["out_offsets"][i + 1])] for i in range(n)]
    streams = [flip_bits(rng, s, 30) if i % 5 == 4 else s for i, s in enumerate(streams)]
    decoders = [oracle.new_decoder(table) for _ in range(n)]
    pos = np.zeros(n, dtype=np.int64)
    fed = np.zeros(n, dtype=np.int64)
    done = np.zeros(n, dtype=bool)
    state = (np.zeros(n, np.uint64), np.zeros(n, np.uint8))
    rounds = 0
    while not done.all():
        rounds += 1
        assert rounds < 5000
        live = np.flatnonzero(~done)
        for i in live:
            if pos[i] == fed[i]:
                fed[i] = min(len(streams[i]), fed[i] + int(rng.integers(1, 8)))
        chunks = [streams[i][pos[i]:fed[i]] for i in live]
        data, in_off = _csr(chunks)
        caps = rng.integers(1, 41, size=len(live)).astype(np.uint64)
        slots = np.zeros(len(live), dtype=np.uint64)
        slots[1:] = np.cumsum(caps)[:-1]
        got = ctx.decode(data, in_off, out_capacity=int(caps.sum()) + 8, out_offsets=slots, out_caps=caps,
                         state=(state[0][live], state[1][live]))
        for j, i in enumerate(live):
            cap, a = int(caps[j]), int(slots[j])
            out = np.zeros(cap, dtype=np.uint8)
            rc, used, olen = oracle.decode_call(decoders[i], chunks[j], out, 0, cap)
            what = "stream %d round %d" % (i, rounds)
            assert (int(got["status"][j]), int(got["consumed"][j]), int(got["out_lens"][j])) == (rc, used, olen), what
            assert np.array_equal(got["out"][a:a + olen], out[:olen]), what
            assert int(got["leftover_num_bits"][j]) == decoders[i].num_bits, what
            assert int(got["leftover_working_bits"][j]) == decoders[i].working_bits, what
            pos[i] += used
            state[0][i], state[1][i] = got["leftover_working_bits"][j], got["leftover_num_bits"][j]
            if rc not in (OK, SHORT_BUFFER) or (rc == OK and fed[i] == len(streams[i]) and pos[i] == fed[i]):
                done[i] = True
