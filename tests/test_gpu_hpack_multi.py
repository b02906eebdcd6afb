"""HPACK string literals and header blocks over several contexts: the _multi entry points of hpack_string_batch.h and
hpack_header_block_batch.h.

Every case runs the multi call and the single-context call on ctxs[0] with the same inputs and the same output arrays,
each followed by guard octets, and compares return value, error and every array the header defines for that outcome;
the guards must be untouched. Some cases are compared with the oracles too. Contexts: two and three on device 0, and
one per device when there are two devices or more.
CPU part (-m "not gpu"): the argument errors that need no device (no context array, no contexts, a NULL context)."""
import ctypes as C

import numpy as np
import pytest

import hpack_records_oracle as rec
import test_hpack_header_blocks as base
import test_hpack_literals as literals

blk, lit = rec.blk, rec.lit
I, INC, WO, NV, SU, AUTO = rec.INDEXED, rec.INCREMENTAL, rec.WITHOUT, rec.NEVER, rec.SIZE_UPDATE, rec.AUTO
MODES = [lit.SMALLEST, lit.NEVER, lit.ALWAYS]
GUARD = 64  # octets behind every output array
FILL = 0xA5


def _ptr(a):
    return a.ctypes.data


def _guarded(count, dtype):
    a = np.empty(count + GUARD // np.dtype(dtype).itemsize, dtype)
    a.view(np.uint8)[:] = FILL
    return a


def _lists(n, fo, kind, index, never, strings, so, field_capacity=0, strings_capacity=0, capi=None):
    return capi.aws_hpack_header_lists(n, _ptr(fo), field_capacity, None if kind is None else _ptr(kind),
                                       None if index is None else _ptr(index), None if never is None else _ptr(never),
                                       None if strings is None else _ptr(strings), strings_capacity, _ptr(so))


class Calls:
    """The five host-pointer calls on one target (a BatchContext, or a list of them for the _multi forms). Each returns
    (error, {name: (array, entries the call may write)}); the arrays are fresh and guarded."""

    def __init__(self, capi, **how):
        self.capi, self.how = capi, how  # how: n_ctx, library (hpack_host_call)

    def _call(self, target, name, *args):
        return self.capi.hpack_host_call(target, name, *args, **self.how)

    def string_encode(self, target, data, offs, mode, cap):
        n = len(offs) - 1
        out, out_off = _guarded(cap, np.uint8), _guarded(n + 1, np.uint64)
        err = self._call(target, "aws_hpack_string_encode_batch", n, _ptr(data), _ptr(offs), mode, _ptr(out),
                         cap, _ptr(out_off))
        return err, {"out": (out, cap), "out_offsets": (out_off, n + 1)}

    def string_decode(self, target, data, offs, cap):
        n = len(offs) - 1
        out, out_off, status = _guarded(cap, np.uint8), _guarded(n + 1, np.uint64), _guarded(n, np.int32)
        err = self._call(target, "aws_hpack_string_decode_batch", n, _ptr(data), _ptr(offs), _ptr(out), cap,
                         _ptr(out_off), _ptr(status))
        return err, {"out": (out, cap), "out_offsets": (out_off, n + 1), "status": (status, n)}

    def block_decode(self, target, data, offs, field_capacity, strings_capacity):
        n = len(offs) - 1
        a = {"field_offsets": (_guarded(n + 1, np.uint64), n + 1), "status": (_guarded(n, np.int32), n),
             "field_kind": (_guarded(field_capacity, np.uint8), field_capacity),
             "field_index": (_guarded(field_capacity, np.uint64), field_capacity),
             "string_offsets": (_guarded(2 * field_capacity + 1, np.uint64), 2 * field_capacity + 1),
             "strings": (_guarded(strings_capacity, np.uint8), strings_capacity)}
        lists = _lists(n, a["field_offsets"][0], a["field_kind"][0], a["field_index"][0], None, a["strings"][0],
                       a["string_offsets"][0], field_capacity, strings_capacity, self.capi)
        err = self._call(target, "aws_hpack_header_block_decode_batch", n, _ptr(data), _ptr(offs),
                         C.byref(lists), _ptr(a["status"][0]))
        return err, a

    def block_encode(self, target, lists_in, mode, cap):
        fo, strings, so, never = lists_in
        n = len(fo) - 1
        out, out_off = _guarded(cap, np.uint8), _guarded(n + 1, np.uint64)
        lists = _lists(n, fo, None, None, never, strings, so, capi=self.capi)
        err = self._call(target, "aws_hpack_header_block_encode_batch", C.byref(lists), mode, _ptr(out), cap,
                         _ptr(out_off))
        return err, {"out": (out, cap), "out_offsets": (out_off, n + 1)}

    def records_encode(self, target, records_in, mode, cap):
        fo, kind, index, strings, so, never = records_in
        n = len(fo) - 1
        out, out_off, status = _guarded(cap, np.uint8), _guarded(n + 1, np.uint64), _guarded(n, np.int32)
        lists = _lists(n, fo, kind, index, never, strings, so, capi=self.capi)
        err = self._call(target, "aws_hpack_header_block_encode_records_batch", C.byref(lists), mode,
                         _ptr(out), cap, _ptr(out_off), _ptr(status))
        return err, {"out": (out, cap), "out_offsets": (out_off, n + 1), "status": (status, n)}


def _defined(err, arrays):
    """The arrays (and how many entries) the header defines for this outcome: AWS_ERROR_SHORT_BUFFER leaves offsets and
    status complete, and string_offsets too when the fields fit."""
    if err != lit.SHORT_BUFFER:
        return {name: count for name, (_, count) in arrays.items()}
    keep = {name: count for name, (_, count) in arrays.items() if name in ("out_offsets", "field_offsets", "status")}
    if "field_offsets" in arrays:
        fields = int(arrays["field_offsets"][0][arrays["field_offsets"][1] - 1])
        if fields <= arrays["field_kind"][1]:
            keep["string_offsets"] = 2 * fields + 1
    return keep


def same(call, ctxs, *args):
    """Runs `call` on ctxs[0] and over ctxs; asserts the same outcome and returns it (error, arrays trimmed to what
    the call may write)."""
    want_err, want = call(ctxs[0], *args)
    got_err, got = call(list(ctxs), *args)
    assert got_err == want_err
    for name, (array, count) in list(want.items()) + list(got.items()):
        assert (array[count:].view(np.uint8) == FILL).all(), "%s written past its capacity" % name
    for name, count in _defined(want_err, want).items():
        a, b = want[name][0][:count], got[name][0][:count]
        assert np.array_equal(a, b), (name, np.flatnonzero(a != b)[:10])
    return got_err, {name: array[:count] for name, (array, count) in got.items()}


# ------------------------------------------------------------------------------------------------ inputs
def _batch(items):
    offs = np.zeros(len(items) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(x) for x in items])
    return np.frombuffer(b"".join(bytes(x) for x in items), dtype=np.uint8), offs


def _damaged_literals(literal_oracle, rng, n):
    """Framed literals, every 5th damaged in one of five ways: the damage is spread over the whole batch, so every
    shard gets some."""
    data, offs = literals._strings(rng, n, 160)
    framed, f_offs = literal_oracle.encode_batch(data, offs, lit.SMALLEST)
    items = [bytearray(framed[int(f_offs[i]):int(f_offs[i + 1])]) for i in range(n)]
    for k, i in enumerate(range(2, n, 5)):
        it, kind = items[i], k % 5
        if kind == 0 and len(it) > 1:
            del it[-1]                                      # cut short
        elif kind == 1:
            it.append(0x00)                                 # octets left over
        elif kind == 2 and it[0] & 0x80 and (it[0] & 0x7f) < 126:
            it[0] += 1
            it.append(0xFF)                                 # a whole octet of padding
        elif kind == 3:
            items[i] = bytearray([0x7f, 0x80, 0x80])        # an unfinished length
        else:
            items[i] = bytearray([0xff] + [0xff] * 10 + [0x01])  # a length beyond 62 bits
    return _batch(items)


def _mixed_blocks(block_oracle, rng, n):
    """Random blocks of all five kinds, the malformed blocks of test_hpack_header_blocks spread over the batch, the RFC
    7541 Appendix C blocks and empty blocks."""
    blocks = [block_oracle.random_block(rng, base._any_bytes)[0] for _ in range(n)]
    for extra in ([b for b, _ in base._malformed_blocks(block_oracle)],
                  [bytes.fromhex(h) for h, _ in base.RFC7541_BLOCKS.values()] + [b"", b""]):
        for j, b in enumerate(extra):
            blocks.insert(((2 * j + 1) * len(blocks)) // (2 * len(extra)), b)
    return _batch(blocks)


def _records(block_oracle, rng, n, mode):
    """Records a decode returns (dynamic indices, size updates, every kind), some fields turned AUTO, never-indexed
    flags, and invalid record lists in several places."""
    blocks = [block_oracle.random_block(rng, base._any_bytes, mode=mode)[0] for _ in range(n)]
    data, offs = _batch(blocks)
    d = block_oracle.decode_batch(data, offs)
    nf = int(d["field_offsets"][-1])
    kinds, index = d["field_kind"].copy(), d["field_index"].copy()
    kinds[(rng.random(nf) < 0.2) & (kinds != SU)] = AUTO
    lists = [[(int(kinds[f]), int(index[f]), bytes(d["strings"][int(d["string_offsets"][2 * f]):int(d["string_offsets"][2 * f + 1])]),
               bytes(d["strings"][int(d["string_offsets"][2 * f + 1]):int(d["string_offsets"][2 * f + 2])]))
              for f in range(int(d["field_offsets"][i]), int(d["field_offsets"][i + 1]))] for i in range(n)]
    bad = [[(6, 1, b"", b"")], [(I, 0, b"", b"")], [(I, 2, b"", b""), (SU, 4096, b"", b"")],
           [(SU, (1 << 64) - 1, b"", b"")], [(WO, 15 + (1 << 63), b"", b"v")]]
    for j, b in enumerate(bad * 2):
        lists.insert((j * len(lists)) // (2 * len(bad)) + 1, b)
    fo, kind, idx, strings, so = rec.records_batch(lists)
    never = (rng.random(len(kind)) < 0.15).astype(np.uint8)
    return fo, kind, idx, strings, so, never


# ------------------------------------------------------------------------------------------------ CPU
def test_argument_errors_without_a_device(pkg, product):
    """ctxs == NULL, n_ctx == 0 and a NULL context fail with AWS_ERROR_INVALID_ARGUMENT in all five calls, before anything
    is written."""
    capi = pkg.capi
    data, offs = np.frombuffer(bytes.fromhex("8286"), np.uint8), np.array([0, 1, 2], np.uint64)
    lists_in = (np.array([0, 1], np.uint64), np.frombuffer(b"ab", np.uint8), np.array([0, 1, 2], np.uint64), None)
    records_in = lists_in[:1] + (np.array([I], np.uint8), np.array([2], np.uint64)) + lists_in[1:]
    for target, n_ctx in ((None, 2), ([None, None], 0), ([None], 1), ([None, None], 2)):
        calls = Calls(capi, n_ctx=n_ctx, library=product)
        for err, arrays in (calls.string_encode(target, data, offs, lit.SMALLEST, 16),
                            calls.string_decode(target, data, offs, 16),
                            calls.block_decode(target, data, offs, 4, 64),
                            calls.block_encode(target, lists_in, lit.SMALLEST, 16),
                            calls.records_encode(target, records_in, lit.SMALLEST, 16)):
            assert err == capi.AWS_ERROR_INVALID_ARGUMENT
            for name, (array, _) in arrays.items():
                assert (array.view(np.uint8) == FILL).all(), name


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def literal_oracle(oracle, oracle_tables):
    return lit.LiteralOracle(oracle, oracle_tables["hpack"])


@pytest.fixture(scope="module")
def block_oracle(oracle, oracle_tables):
    return rec.RecordsOracle(lit.LiteralOracle(oracle, oracle_tables["hpack"]))


@pytest.fixture(scope="module")
def context_sets(pkg, coders):
    made = {}

    def get(name):
        if name not in made:
            import torch
            if name == "one_per_device":
                if torch.cuda.device_count() < 2:
                    pytest.skip("one device")
                devices = list(range(torch.cuda.device_count()))
            else:
                devices = [0] * {"two_on_device_0": 2, "three_on_device_0": 3}[name]
            made[name] = [pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=d) for d in devices]
        return made[name]

    yield get
    for contexts in made.values():
        for c in contexts:
            c.close()


@pytest.fixture(params=["two_on_device_0", "three_on_device_0", "one_per_device"])
def ctxs(request, context_sets):
    return context_sets(request.param)


@pytest.fixture(scope="module")
def calls(pkg):
    return Calls(pkg.capi)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_string_encode(ctxs, calls, literal_oracle, mode):
    rng = np.random.default_rng(10 + mode)
    data, offs = literals._strings(rng, 3000, 200)
    want, want_offs = literal_oracle.encode_batch(data, offs, mode)
    err, got = same(calls.string_encode, ctxs, data, offs, mode, len(want) + 64)
    assert err == 0 and np.array_equal(got["out_offsets"], want_offs) and np.array_equal(got["out"][:len(want)], want)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["one_kernel", "passes"])
def test_string_decode_with_malformed_literals(ctxs, calls, literal_oracle, monkeypatch, route):
    if route == "passes":
        monkeypatch.setenv("AWS_HUFFMAN_HPACK_PASSES", "1")
    framed, offs = _damaged_literals(literal_oracle, np.random.default_rng(11), 2500)
    want, want_offs, want_status = literal_oracle.decode_batch(framed, offs)
    err, got = same(calls.string_decode, ctxs, framed, offs, len(want) + 4096)
    assert err == 0 and np.array_equal(got["status"], want_status) and np.array_equal(got["out_offsets"], want_offs)
    assert np.array_equal(got["out"][:len(want)], want)
    bad = np.flatnonzero(want_status)
    assert {lit.SHORT_BUFFER, lit.INVALID_ARGUMENT, lit.INVALID_PADDING} <= set(want_status[bad].tolist())
    assert bad.min() < len(want_status) // 8 and bad.max() > len(want_status) * 7 // 8


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["one_kernel", "passes"])
def test_block_decode(ctxs, calls, block_oracle, monkeypatch, route):
    if route == "passes":
        monkeypatch.setenv("AWS_HUFFMAN_HPACK_PASSES", "1")
    data, offs = _mixed_blocks(block_oracle, np.random.default_rng(12), 1500)
    want = block_oracle.decode_batch(data, offs)
    n_in = len(data)
    err, got = same(calls.block_decode, ctxs, data, offs, n_in, 28 * n_in)
    assert err == 0
    base.assert_decode_matches(got, want)
    assert set(want["field_kind"]) == {I, INC, WO, NV, SU} and (want["field_index"][want["field_kind"] == I] >= 62).any()
    bad = np.flatnonzero(want["status"])
    assert bad.min() < len(offs) // 8 and bad.max() > len(offs) * 7 // 8


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_block_encode(ctxs, calls, block_oracle, mode):
    fo, strings, so, never = base._random_lists(np.random.default_rng(13 + mode), 800)
    want, want_offs = block_oracle.encode_batch(fo, strings, so, never, mode)
    err, got = same(calls.block_encode, ctxs, (fo, strings, so, never), mode, len(want) + 64)
    assert err == 0 and np.array_equal(got["out_offsets"], want_offs) and np.array_equal(got["out"][:len(want)], want)
    assert never.any()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_records_encode(ctxs, calls, block_oracle, mode):
    fo, kind, index, strings, so, never = _records(block_oracle, np.random.default_rng(14 + mode), 1000, mode)
    want, want_offs, want_status = block_oracle.encode_records_batch(fo, kind, index, strings, so, never, mode)
    err, got = same(calls.records_encode, ctxs, (fo, kind, index, strings, so, never), mode, len(want) + 64)
    assert err == 0 and np.array_equal(got["status"], want_status) and np.array_equal(got["out_offsets"], want_offs)
    assert np.array_equal(got["out"][:len(want)], want)
    assert {I, INC, WO, NV, SU, AUTO} <= set(kind.tolist()) and (index[kind == I] >= 62).any()
    bad = np.flatnonzero(want_status)
    assert len(bad) >= 10 and bad.min() < len(fo) // 8 and bad.max() > len(fo) * 6 // 8


def _shapes(block_oracle):
    """(name, literal strings, header blocks): no items, fewer items than contexts, one item holding almost every
    octet, empty items."""
    rng = np.random.default_rng(15)
    big = base._text(rng, 300_000)
    huge = b"\x10\x00" + lit.encode_integer(len(big), 7) + big  # never indexed, literal name "", a 300 KB value
    small = [bytes.fromhex("82"), b"", bytes.fromhex("418cf1e3c2e5f23a6ba0ab90f4ff")]
    return [("none", [], []),
            ("one", [b"custom-key"], small[:1]),
            ("two", [b"", b"www.example.com"], small[:2]),
            ("one_huge", [b"a", big, b"", b"xyz"], [small[0], huge, b"", bytes.fromhex("828684")]),
            ("all_empty", [b""] * 7, [b""] * 7)]


@pytest.mark.gpu
def test_shapes(ctxs, calls, block_oracle, literal_oracle):
    for n_ctx in sorted({1, len(ctxs)}):
        sub = ctxs[:n_ctx]
        for name, strings, blocks in _shapes(block_oracle):
            data, offs = _batch(strings)
            want, want_offs = literal_oracle.encode_batch(data, offs, lit.SMALLEST)
            err, enc = same(calls.string_encode, sub, data, offs, lit.SMALLEST, len(want) + 16)
            assert err == 0 and np.array_equal(enc["out_offsets"], want_offs), name
            err, dec = same(calls.string_decode, sub, want, want_offs, len(data) + 16)
            assert err == 0 and np.array_equal(dec["out"][:len(data)], data) and not dec["status"].any(), name
            bdata, boffs = _batch(blocks)
            d_err, d = same(calls.block_decode, sub, bdata, boffs, len(bdata), 28 * len(bdata))
            assert d_err == 0, name
            base.assert_decode_matches(d, block_oracle.decode_batch(bdata, boffs))
            nf = int(d["field_offsets"][-1])
            lists_in = (d["field_offsets"].copy(), d["strings"][:int(d["string_offsets"][2 * nf])].copy(),
                        d["string_offsets"][:2 * nf + 1].copy(), np.zeros(max(nf, 1), np.uint8))
            err, e = same(calls.block_encode, sub, lists_in, lit.SMALLEST, 2 * len(bdata) + 64)
            assert err == 0, name
            kind, index = np.zeros(max(nf, 1), np.uint8), np.zeros(max(nf, 1), np.uint64)
            kind[:nf], index[:nf] = d["field_kind"][:nf], d["field_index"][:nf]
            records_in = (lists_in[0], kind, index) + lists_in[1:]
            err, r = same(calls.records_encode, sub, records_in, lit.NEVER, 2 * len(bdata) + 64)
            assert err == 0 and not r["status"].any(), name
            if name == "one_huge":  # the raw literals give the block back
                assert bytes(r["out"][:int(r["out_offsets"][-1])]) == bytes(bdata)


@pytest.mark.gpu
def test_capacities_exact_and_one_short(ctxs, calls, block_oracle, literal_oracle):
    """At the exact size every call succeeds; one short, the same AWS_ERROR_SHORT_BUFFER with the same complete arrays
    as the single-context call, and nothing past any capacity (same() checks the guards)."""
    rng = np.random.default_rng(16)
    data, offs = literals._strings(rng, 2000, 120)
    want, want_offs = literal_oracle.encode_batch(data, offs, lit.ALWAYS)
    for short in (0, 1):
        expect = lit.SHORT_BUFFER if short else 0
        assert same(calls.string_encode, ctxs, data, offs, lit.ALWAYS, len(want) - short)[0] == expect
        assert same(calls.string_decode, ctxs, want, want_offs, len(data) - short)[0] == expect
    bdata, boffs = _mixed_blocks(block_oracle, rng, 600)
    d = block_oracle.decode_batch(bdata, boffs)
    nf, ns = int(d["field_offsets"][-1]), len(d["strings"])
    for fcap, scap, expect in ((nf, ns, 0), (nf - 1, ns, lit.SHORT_BUFFER), (nf, ns - 1, lit.SHORT_BUFFER)):
        err, got = same(calls.block_decode, ctxs, bdata, boffs, fcap, scap)
        assert err == expect and np.array_equal(got["field_offsets"], d["field_offsets"])
        assert np.array_equal(got["status"], d["status"])
    lists_in = (d["field_offsets"], d["strings"], d["string_offsets"], (rng.random(nf) < 0.2).astype(np.uint8))
    total = int(same(calls.block_encode, ctxs, lists_in, lit.SMALLEST, 1 << 22)[1]["out_offsets"][-1])
    for cap, expect in ((total, 0), (total - 1, lit.SHORT_BUFFER)):
        assert same(calls.block_encode, ctxs, lists_in, lit.SMALLEST, cap)[0] == expect
    records_in = _records(block_oracle, rng, 600, lit.SMALLEST)
    want, want_offs, want_status = block_oracle.encode_records_batch(*records_in[:5], records_in[5], lit.SMALLEST)
    for cap, expect in ((len(want), 0), (len(want) - 1, lit.SHORT_BUFFER)):
        err, got = same(calls.records_encode, ctxs, records_in, lit.SMALLEST, cap)
        assert err == expect and np.array_equal(got["out_offsets"], want_offs) and np.array_equal(got["status"], want_status)


@pytest.mark.gpu
def test_argument_errors(pkg, ctxs, calls):
    """Decreasing offsets, a NULL context among real ones, no contexts: the single call's error, or
    AWS_ERROR_INVALID_ARGUMENT; nothing written."""
    capi = pkg.capi
    data = np.frombuffer(bytes.fromhex("828684"), np.uint8)
    down = np.array([0, 2, 1, 3], np.uint64)
    assert same(calls.block_decode, ctxs, data, down, 8, 256)[0] == capi.AWS_ERROR_INVALID_ARGUMENT
    strings = np.frombuffer(b"abcdefgh", np.uint8)
    for fo, so in ((np.array([0, 2, 1], np.uint64), np.array([0, 2, 4, 6, 8], np.uint64)),
                   (np.array([0, 2], np.uint64), np.array([0, 2, 6, 4, 8], np.uint64))):
        assert same(calls.block_encode, ctxs, (fo, strings, so, None), lit.NEVER, 64)[0] == capi.AWS_ERROR_INVALID_ARGUMENT
    offs = np.array([0, 1, 2, 3], np.uint64)
    for target in (list(ctxs) + [None], [None] + list(ctxs)):
        for err, arrays in (calls.string_encode(target, data, offs, lit.NEVER, 64), calls.string_decode(target, data, offs, 64),
                            calls.block_decode(target, data, offs, 8, 256)):
            assert err == capi.AWS_ERROR_INVALID_ARGUMENT
            assert all((a.view(np.uint8) == FILL).all() for a, _ in arrays.values())
    assert calls.string_encode(list(ctxs), data, offs, 3, 64)[0] == capi.AWS_ERROR_INVALID_ARGUMENT
