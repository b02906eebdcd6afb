"""HPACK header blocks (RFC 7541 section 6, Appendix A; include/aws/compression/hpack_header_block_batch.h).

CPU part (-m "not gpu"): the block oracle (oracle/hpack_header_block_oracle.py) against RFC 7541 Appendix C: every
block decodes to the RFC's representations, and a dynamic table kept here rebuilds the RFC's header lists from the
records alone (so the records are enough for a caller that keeps the table); the encoder rules; the header compiles;
no device means no result.
GPU part: aws_hpack_header_block_decode_batch / _encode_batch through the C ABI against that oracle, array for array,
including malformed blocks, both literal routes, every Huffman mode and the capacity contract."""
import ctypes as C
import importlib.util
import os
import subprocess
from collections import deque

import numpy as np
import pytest

import refcodec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(name, *path):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, *path))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module


blk = _load("hpack_header_block_oracle", "oracle", "hpack_header_block_oracle.py")
lit = blk.lit
I, INC, WO, NV, SU = blk.INDEXED, blk.INCREMENTAL, blk.WITHOUT, blk.NEVER, blk.SIZE_UPDATE

# RFC 7541 Appendix C header blocks and their representations: (kind, index, literal name or None, literal value)
RFC7541_BLOCKS = {
    "C.2.1": ("400a637573746f6d2d6b65790d637573746f6d2d686561646572", [(INC, 0, b"custom-key", b"custom-header")]),
    "C.2.2": ("040c2f73616d706c652f70617468", [(WO, 4, None, b"/sample/path")]),
    "C.2.3": ("100870617373776f726406736563726574", [(NV, 0, b"password", b"secret")]),
    "C.2.4": ("82", [(I, 2, None, None)]),
    "C.3.1": ("828684410f7777772e6578616d706c652e636f6d",
              [(I, 2, None, None), (I, 6, None, None), (I, 4, None, None), (INC, 1, None, b"www.example.com")]),
    "C.3.2": ("828684be58086e6f2d6361636865",
              [(I, 2, None, None), (I, 6, None, None), (I, 4, None, None), (I, 62, None, None),
               (INC, 24, None, b"no-cache")]),
    "C.3.3": ("828785bf400a637573746f6d2d6b65790c637573746f6d2d76616c7565",
              [(I, 2, None, None), (I, 7, None, None), (I, 5, None, None), (I, 63, None, None),
               (INC, 0, b"custom-key", b"custom-value")]),
    "C.5.1": ("4803333032580770726976617465611d4d6f6e2c203231204f637420323031332032303a31333a323120474d546e1768"
              "747470733a2f2f7777772e6578616d706c652e636f6d",
              [(INC, 8, None, b"302"), (INC, 24, None, b"private"), (INC, 33, None, b"Mon, 21 Oct 2013 20:13:21 GMT"),
               (INC, 46, None, b"https://www.example.com")]),
    "C.6.2": ("4883640effc1c0bf", [(INC, 8, None, b"307"), (I, 65, None, None), (I, 64, None, None), (I, 63, None, None)]),
    "C.6.3": ("88c16196d07abe941054d444a8200595040b8166e084a62d1bffc05a839bd9ab77ad94e7821dd7f2e6c7b335dfdfcd5b3960d5af"
              "27087f3672c1ab270fb5291f9587316065c003ed4ee5b1063d5007",
              [(I, 8, None, None), (I, 65, None, None), (INC, 33, None, b"Mon, 21 Oct 2013 20:13:22 GMT"),
               (I, 64, None, None), (INC, 26, None, b"gzip"),
               (INC, 55, None, b"foo=ASDJKHQKBZXOQWEOPIUAXQWEOIU; max-age=3600; version=1")]),
}
# C.4.x / C.6.1 are C.3.x / C.5.1 with Huffman-coded literals: the same representations
RFC7541_BLOCKS["C.4.1"] = ("828684418cf1e3c2e5f23a6ba0ab90f4ff", RFC7541_BLOCKS["C.3.1"][1])
RFC7541_BLOCKS["C.4.2"] = ("828684be5886a8eb10649cbf", RFC7541_BLOCKS["C.3.2"][1])
RFC7541_BLOCKS["C.4.3"] = ("828785bf408825a849e95ba97d7f8925a849e95bb8e8b4bf", RFC7541_BLOCKS["C.3.3"][1])
RFC7541_BLOCKS["C.6.1"] = ("488264025885aec3771a4b6196d07abe941054d444a8200595040b8166e082a62d1bff6e919d29ad171863c78f0b97"
                           "c8e9ae82ae43d3", RFC7541_BLOCKS["C.5.1"][1])

# RFC 7541's decoded header lists (C.3 / C.4 requests, C.5 / C.6 responses)
_DATE1, _DATE2, _LOC = b"Mon, 21 Oct 2013 20:13:21 GMT", b"Mon, 21 Oct 2013 20:13:22 GMT", b"https://www.example.com"
REQUESTS = [
    [(b":method", b"GET"), (b":scheme", b"http"), (b":path", b"/"), (b":authority", b"www.example.com")],
    [(b":method", b"GET"), (b":scheme", b"http"), (b":path", b"/"), (b":authority", b"www.example.com"),
     (b"cache-control", b"no-cache")],
    [(b":method", b"GET"), (b":scheme", b"https"), (b":path", b"/index.html"), (b":authority", b"www.example.com"),
     (b"custom-key", b"custom-value")],
]
RESPONSES = [
    [(b":status", b"302"), (b"cache-control", b"private"), (b"date", _DATE1), (b"location", _LOC)],
    [(b":status", b"307"), (b"cache-control", b"private"), (b"date", _DATE1), (b"location", _LOC)],
    [(b":status", b"200"), (b"cache-control", b"private"), (b"date", _DATE2), (b"location", _LOC),
     (b"content-encoding", b"gzip"), (b"set-cookie", b"foo=ASDJKHQKBZXOQWEOPIUAXQWEOIU; max-age=3600; version=1")],
]


def expected_records(reps):
    return [(kind, index) + blk.field_strings(kind, index, name or b"", value or b"") for kind, index, name, value in reps]


class DynamicTable:
    """A caller's dynamic table (RFC 7541 section 2.3.2 / 4), driven only by the decoder's records."""

    def __init__(self, max_size):
        self.max_size, self.size, self.entries = max_size, 0, deque()

    def _evict(self):
        while self.size > self.max_size:
            name, value = self.entries.pop()
            self.size -= 32 + len(name) + len(value)

    def resolve(self, records):
        headers = []
        for kind, index, name, value in records:
            if kind == SU:
                self.max_size = index
                self._evict()
                continue
            if index > 61:
                entry = self.entries[index - 62]
                name, value = entry if kind == I else (entry[0], value)
            headers.append((name, value))
            if kind == INC:
                self.entries.appendleft((name, value))
                self.size += 32 + len(name) + len(value)
                self._evict()
        return headers


@pytest.fixture(scope="module")
def block_oracle(oracle, oracle_tables):
    return blk.BlockOracle(lit.LiteralOracle(oracle, oracle_tables["hpack"]))


def _text(rng, length):
    return bytes(rng.choice(np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789-_/:;=, ", np.uint8), size=length))


def _any_bytes(rng, length):
    return rng.integers(0, 256, size=length, dtype=np.uint8).tobytes() if rng.random() < 0.2 else _text(rng, length)


def _random_lists(rng, n, max_fields=10):
    """Header lists mixing exact static entries, static names and custom names (empty strings too)."""
    names = [n for n, _ in blk.STATIC_TABLE] + [b"x-custom", b"custom-key", b"", b"X-Upper"]
    fields, never = [], []
    offs = [0]
    for _ in range(n):
        for _ in range(int(rng.integers(0, max_fields + 1))):
            r = rng.random()
            if r < 0.25:
                fields += list(blk.STATIC_TABLE[int(rng.integers(0, 61))])
            else:
                fields += [names[int(rng.integers(0, len(names)))] if r < 0.8 else _text(rng, int(rng.integers(1, 20))),
                           _any_bytes(rng, int(rng.choice([0, 3, 17, 60, 130])))]
            never.append(1 if rng.random() < 0.15 else 0)
        offs.append(len(never))
    string_offsets = np.zeros(len(fields) + 1, dtype=np.uint64)
    string_offsets[1:] = np.cumsum([len(s) for s in fields])
    return (np.array(offs, dtype=np.uint64), np.frombuffer(b"".join(fields), dtype=np.uint8), string_offsets,
            np.array(never, dtype=np.uint8))


def _batch(blocks):
    offs = np.zeros(len(blocks) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(b) for b in blocks])
    return np.frombuffer(b"".join(blocks), dtype=np.uint8), offs


# ------------------------------------------------------------------------------------------------ CPU
def test_oracle_decodes_rfc7541_appendix_c_blocks(block_oracle):
    for name, (hexed, reps) in RFC7541_BLOCKS.items():
        assert block_oracle.decode_block(bytes.fromhex(hexed)) == (lit.OK, expected_records(reps)), name


@pytest.mark.parametrize("blocks,max_size,lists,sizes", [
    (["C.3.1", "C.3.2", "C.3.3"], 4096, REQUESTS, [57, 110, 164]),
    (["C.4.1", "C.4.2", "C.4.3"], 4096, REQUESTS, [57, 110, 164]),
    (["C.5.1", "C.6.2", "C.6.3"], 256, RESPONSES, [222, 222, 215]),
    (["C.6.1", "C.6.2", "C.6.3"], 256, RESPONSES, [222, 222, 215]),
])
def test_records_are_enough_to_rebuild_the_rfc_header_lists(block_oracle, blocks, max_size, lists, sizes):
    """C.6.2's c1 is cache-control: private because C.6.1's :status 302 was evicted (256-octet table)."""
    table = DynamicTable(max_size)
    for name, want, size in zip(blocks, lists, sizes):
        st, records = block_oracle.decode_block(bytes.fromhex(RFC7541_BLOCKS[name][0]))
        assert st == lit.OK
        assert table.resolve(records) == want, name
        assert table.size == size, name


def test_oracle_encoder_rules(block_oracle):
    enc = block_oracle.encode_field
    assert enc(b":method", b"GET") == bytes.fromhex("82")                              # C.2.4: exact static match
    assert enc(b"cache-control", b"no-cache", mode=lit.NEVER) == bytes.fromhex("0f09") + b"\x08no-cache"  # index 24
    assert enc(b"cache-control", b"no-cache", True, lit.NEVER) == bytes.fromhex("1f09") + b"\x08no-cache"
    assert enc(b":method", b"GET", True, lit.NEVER) == bytes.fromhex("12") + b"\x03GET"  # never-indexed beats exact
    assert enc(b":path", b"/sample/path", mode=lit.NEVER) == bytes.fromhex(RFC7541_BLOCKS["C.2.2"][0])  # C.2.2
    assert enc(b"password", b"secret", True, lit.NEVER) == bytes.fromhex(RFC7541_BLOCKS["C.2.3"][0])    # C.2.3
    assert enc(b"custom-key", b"custom-header", mode=lit.NEVER) == bytes.fromhex("00") + bytes.fromhex(
        RFC7541_BLOCKS["C.2.1"][0])[1:]
    assert enc(b":status", b"302", mode=lit.NEVER) == bytes.fromhex("08") + b"\x03302"  # lowest :status index
    assert enc(b"www-authenticate", b"x", mode=lit.NEVER) == bytes.fromhex("0f2e0178")  # index 61
    assert enc(b"www-authenticate", b"") == bytes.fromhex("bd")                        # empty values match too
    assert enc(b":authority", b"", mode=lit.NEVER) == bytes.fromhex("81")              # index 1 is an exact match


def test_oracle_encode_then_decode_is_the_identity(block_oracle):
    rng = np.random.default_rng(3)
    fo, strings, so, never = _random_lists(rng, 60)
    for mode in (lit.SMALLEST, lit.NEVER, lit.ALWAYS):
        data, offs = block_oracle.encode_batch(fo, strings, so, never, mode)
        got = block_oracle.decode_batch(data, offs)
        assert not got["status"].any()
        assert np.array_equal(got["field_offsets"], fo)
        assert np.array_equal(got["string_offsets"], so) and np.array_equal(got["strings"], strings)
        assert set(got["field_kind"][never == 1]) <= {NV} and I not in set(got["field_kind"][never == 1])


def test_random_writer_emits_every_kind_and_its_records(block_oracle):
    rng = np.random.default_rng(8)
    kinds = set()
    for _ in range(300):
        block, records = block_oracle.random_block(rng, _any_bytes)
        assert block_oracle.decode_block(block) == (lit.OK, records)
        kinds |= {r[0] for r in records}
    assert kinds == {I, INC, WO, NV, SU}


def test_header_compiles_as_c_and_cxx(pkg, tmp_path):
    inc = [a for d in pkg._build.INCLUDES for a in ("-I", d)]
    for compiler, ext, std in (("gcc", "c", "-std=c99"), ("g++", "cpp", "-std=c++14")):
        src = tmp_path / ("blocks." + ext)
        src.write_text("#include <aws/compression/hpack_header_block_batch.h>\n"
                       "int main(void){struct aws_hpack_header_lists l; enum aws_hpack_field_kind k = "
                       "AWS_HPACK_FIELD_TABLE_SIZE_UPDATE; (void)l; (void)k; return 0;}\n")
        subprocess.check_call([compiler, std, "-Wall", "-Werror", *inc, "-c", "-o", str(tmp_path / "o.o"), str(src)])


def test_lists_struct_matches_the_header(pkg, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <aws/compression/hpack_header_block_batch.h>\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void){printf("%zu %zu %zu\\n", sizeof(struct aws_hpack_header_lists),'
                   'offsetof(struct aws_hpack_header_lists, strings_capacity),'
                   'offsetof(struct aws_hpack_header_lists, string_offsets));return 0;}\n')
    exe = tmp_path / "layout"
    inc = [a for d in pkg._build.INCLUDES for a in ("-I", d)]
    subprocess.check_call(["gcc", "-std=gnu99", *inc, "-o", str(exe), str(src)])
    t = pkg.capi.aws_hpack_header_lists
    assert subprocess.check_output([str(exe)], text=True).split() == [
        str(C.sizeof(t)), str(t.strings_capacity.offset), str(t.string_offsets.offset)]


def test_no_device_means_no_result(pkg, coders, product):
    """Without a device there is no context (AWS_ERROR_COMPRESSION_DEVICE_FAILURE), and without a context every
    header-block entry point fails with AWS_ERROR_INVALID_ARGUMENT, writing nothing, instead of computing anything
    on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.CodecError) as err:
        pkg.BatchContext(coders.coder("hpack"), device=0)
    assert err.value.code == pkg.AWS_ERROR_COMPRESSION_DEVICE_FAILURE
    L = product.lib
    data = np.frombuffer(bytes.fromhex("82"), np.uint8)
    offs = np.array([0, 1], np.uint64)
    fo, so = np.full(2, 7, np.uint64), np.full(3, 7, np.uint64)
    lists = pkg.capi.aws_hpack_header_lists(1, fo.ctypes.data, 1, None, None, None, None, 0, so.ctypes.data)
    out = np.zeros(8, np.uint8)
    calls = [
        lambda: L.aws_hpack_header_block_decode_batch(None, 1, data.ctypes.data, offs.ctypes.data, C.byref(lists), None),
        lambda: L.aws_hpack_header_block_encode_batch(None, C.byref(lists), 0, out.ctypes.data, 8, offs.ctypes.data),
        lambda: L.aws_hpack_header_block_decode_batch_device(None, 1, data.ctypes.data, offs.ctypes.data, 1,
                                                             C.byref(lists), None, None),
        lambda: L.aws_hpack_header_block_encode_batch_device(None, C.byref(lists), 1, 0, 0, out.ctypes.data, 8,
                                                             offs.ctypes.data, None),
    ]
    for call in calls:
        L.aws_reset_error()
        assert call() == pkg.capi.AWS_OP_ERR
        assert L.aws_last_error() == pkg.capi.AWS_ERROR_INVALID_ARGUMENT
    assert (fo == 7).all() and (so == 7).all() and not out.any()


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def hpack_ctx(pkg, coders):
    ctx = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
    yield ctx
    ctx.close()


def assert_decode_matches(got, want):
    assert np.array_equal(got["status"], want["status"]), np.flatnonzero(got["status"] != want["status"])[:10]
    assert np.array_equal(got["field_offsets"], want["field_offsets"])
    nf = int(want["field_offsets"][-1])
    assert np.array_equal(got["field_kind"][:nf], want["field_kind"])
    assert np.array_equal(got["field_index"][:nf], want["field_index"])
    assert np.array_equal(got["string_offsets"][:2 * nf + 1], want["string_offsets"])
    assert np.array_equal(got["strings"][:len(want["strings"])], want["strings"])


@pytest.mark.gpu
def test_appendix_c_blocks_in_one_batch(hpack_ctx, block_oracle):
    data, offs = _batch([bytes.fromhex(h) for h, _ in RFC7541_BLOCKS.values()])
    got = hpack_ctx.hpack_decode_blocks(data, offs)
    want = block_oracle.decode_batch(data, offs)
    assert_decode_matches(got, want)
    assert not want["status"].any() and int(want["field_offsets"][-1]) == sum(len(r) for _, r in RFC7541_BLOCKS.values())


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["one_kernel", "passes"])
def test_random_blocks_match_oracle(hpack_ctx, block_oracle, monkeypatch, route):
    if route == "passes":
        monkeypatch.setenv("AWS_HUFFMAN_HPACK_PASSES", "1")
    rng = np.random.default_rng(21)
    blocks = [block_oracle.random_block(rng, _any_bytes)[0] for _ in range(1500)] + [b"", b""]
    rng.shuffle(blocks)
    data, offs = _batch(blocks)
    want = block_oracle.decode_batch(data, offs)
    assert_decode_matches(hpack_ctx.hpack_decode_blocks(data, offs), want)
    assert set(want["field_kind"]) == {I, INC, WO, NV, SU} and not want["status"].any()
    assert (want["field_index"][want["field_kind"] == I] >= 62).any()


def _malformed_blocks(block_oracle):
    """(block, status) pairs, one kind of damage each, behind a valid prefix."""
    good = bytes.fromhex("828684")                    # three indexed fields
    huff = bytes.fromhex("418cf1e3c2e5f23a6ba0ab90f4ff")  # :authority www.example.com, Huffman
    bad_pad = bytearray(huff)
    bad_pad[1] += 1
    bad_pad.append(0xFF)                              # a whole octet of padding
    eos = bytearray(huff)
    eos[1] += 4
    eos += b"\xff\xff\xff\xff"                        # EOS with 32 bits or more behind it
    long_int = bytes([0xFF] + [0xFF] * 9 + [0x01])    # ten continuation octets
    return [
        (good + bytes([0xFF, 0x80]), lit.SHORT_BUFFER),          # cut inside an integer
        (good + huff[:-3], lit.SHORT_BUFFER),                    # cut inside a literal
        (good + b"\x04", lit.SHORT_BUFFER),                      # a name index and no value literal
        (good + b"\x80", lit.INVALID_ARGUMENT),                  # index 0
        (good + b"\x3f\xe1\x1f", lit.INVALID_ARGUMENT),          # a size update after a field
        (b"\x20\x3f\xe1\x1f" + good + b"\x20", lit.INVALID_ARGUMENT),  # updates first are fine, a later one is not
        (good + long_int, lit.INVALID_ARGUMENT),                 # an integer over 62 bits
        (good + b"\x04" + long_int, lit.INVALID_ARGUMENT),       # ... as a literal length
        (good + bytes(bad_pad), lit.INVALID_PADDING),            # bad padding
        (good + bytes(eos), lit.UNKNOWN_SYMBOL),                 # EOS inside a payload
        (good + bytes(eos) + b"\x80", lit.UNKNOWN_SYMBOL),       # the Huffman error comes first ...
        (good + bytes(bad_pad) + b"\x3f\xe1\x1f", lit.INVALID_PADDING),
        (good + b"\x80" + bytes(bad_pad), lit.INVALID_ARGUMENT),  # ... unless the structural error does
        # a field that fails after its name literal: that literal's Huffman error comes first
        (b"\x40\x81\xff", lit.INVALID_PADDING),                 # bad name, block ends before the value
        (good + b"\x00\x81\xff\x04", lit.INVALID_PADDING),       # bad name, value literal cut short
        (good + b"\x10\x81\xff" + long_int, lit.INVALID_PADDING),  # bad name, value length over 62 bits
        (good + b"\x00" + bytes(eos[1:]) + b"\x04", lit.UNKNOWN_SYMBOL),  # EOS in the name, value cut short
        (good + b"\x40" + bytes(huff[1:]) + b"\x04", lit.SHORT_BUFFER),  # a good Huffman name, value cut short
        (good + b"\x40\x01a", lit.SHORT_BUFFER),                  # a good raw name, no value
        (good + huff, lit.OK),
        (b"", lit.OK),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["one_kernel", "passes"])
def test_malformed_blocks_report_the_first_error_and_no_fields(hpack_ctx, block_oracle, monkeypatch, route):
    if route == "passes":
        monkeypatch.setenv("AWS_HUFFMAN_HPACK_PASSES", "1")
    cases = _malformed_blocks(block_oracle)
    blocks = [b for b, _ in cases] * 3
    data, offs = _batch(blocks)
    want = block_oracle.decode_batch(data, offs)
    assert list(want["status"][:len(cases)]) == [st for _, st in cases]
    got = hpack_ctx.hpack_decode_blocks(data, offs)
    assert_decode_matches(got, want)
    counts = np.diff(got["field_offsets"].astype(np.int64))
    assert (counts[got["status"] != 0] == 0).all()
    # a batch whose only literal belongs to no field
    alone = hpack_ctx.hpack_decode_blocks(np.frombuffer(b"\x40\x81\xff", np.uint8), np.array([0, 3], np.uint64))
    assert list(alone["status"]) == [lit.INVALID_PADDING] and list(alone["field_offsets"]) == [0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.SMALLEST, lit.NEVER, lit.ALWAYS])
def test_encode_matches_oracle_and_decodes_back(hpack_ctx, block_oracle, mode):
    rng = np.random.default_rng(50 + mode)
    fo, strings, so, never = _random_lists(rng, 800)
    want, want_offs = block_oracle.encode_batch(fo, strings, so, never, mode)
    got = hpack_ctx.hpack_encode_blocks(fo, strings, so, out_capacity=len(want) + 64, mode=mode, never_indexed=never)
    assert np.array_equal(got["out_offsets"], want_offs)
    assert np.array_equal(got["out"][:len(want)], want)
    back = hpack_ctx.hpack_decode_blocks(want, want_offs)
    assert not back["status"].any() and np.array_equal(back["field_offsets"], fo)
    assert np.array_equal(back["string_offsets"][:len(so)], so) and np.array_equal(back["strings"][:len(strings)], strings)
    kinds = back["field_kind"][:len(never)]
    assert (kinds[never == 1] == NV).all() and set(kinds) <= {I, WO, NV} and I in set(kinds)
    # cache-control (index 24) takes a continuation octet under the 4-bit prefix, never-indexed or not
    for flag, head in ((1, "1f09"), (0, "0f09")):
        one = hpack_ctx.hpack_encode_blocks(np.array([0, 1], np.uint64), np.frombuffer(b"cache-controlno-cache", np.uint8),
                                            np.array([0, 13, 21], np.uint64), out_capacity=64, mode=lit.NEVER,
                                            never_indexed=np.array([flag], np.uint8))
        assert bytes(one["out"][:int(one["out_offsets"][1])]) == bytes.fromhex(head) + b"\x08no-cache"


@pytest.mark.gpu
def test_capacity_contract(hpack_ctx, block_oracle, pkg):
    rng = np.random.default_rng(4)
    blocks = [block_oracle.random_block(rng, _text)[0] for _ in range(200)]
    data, offs = _batch(blocks)
    want = block_oracle.decode_batch(data, offs)
    nf, ns = int(want["field_offsets"][-1]), len(want["strings"])
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.hpack_decode_blocks(data, offs, field_capacity=nf - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    assert np.array_equal(err.value.result["field_offsets"], want["field_offsets"])
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.hpack_decode_blocks(data, offs, field_capacity=nf, strings_capacity=ns - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    assert np.array_equal(err.value.result["field_offsets"], want["field_offsets"])
    assert np.array_equal(err.value.result["string_offsets"], want["string_offsets"])
    assert_decode_matches(hpack_ctx.hpack_decode_blocks(data, offs, field_capacity=nf, strings_capacity=ns), want)
    # the documented bounds are tight on the worst block: every octet a field of 28 octets
    worst = np.full(4096, 0x90, np.uint8)
    got = hpack_ctx.hpack_decode_blocks(worst, np.array([0, 4096], np.uint64), field_capacity=4096,
                                        strings_capacity=28 * 4096)
    assert int(got["field_offsets"][-1]) == 4096 and int(got["string_offsets"][-1]) == 28 * 4096
    enc = hpack_ctx.hpack_encode_blocks(want["field_offsets"], want["strings"], want["string_offsets"], out_capacity=1 << 20)
    total = int(enc["out_offsets"][-1])
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.hpack_encode_blocks(want["field_offsets"], want["strings"], want["string_offsets"], out_capacity=total - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    assert np.array_equal(err.value.result["out_offsets"], enc["out_offsets"])
    empty = hpack_ctx.hpack_decode_blocks(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    assert list(empty["field_offsets"]) == [0]
    # decreasing offsets, and encode offsets that do not start at 0, are refused before any kernel reads them
    for call in (lambda: hpack_ctx.hpack_decode_blocks(data, np.array([0, 5, 2, len(data)], np.uint64)),
                 lambda: hpack_ctx.hpack_encode_blocks(np.array([1, 2], np.uint64), np.zeros(8, np.uint8),
                                                       np.array([0, 2, 4, 6, 8], np.uint64), out_capacity=64),
                 lambda: hpack_ctx.hpack_encode_blocks(np.array([0, 1], np.uint64), np.zeros(8, np.uint8),
                                                       np.array([2, 4, 6], np.uint64), out_capacity=64),
                 lambda: hpack_ctx.hpack_encode_blocks(np.array([0, 2, 1], np.uint64), want["strings"],
                                                       want["string_offsets"][:5], out_capacity=1 << 16),
                 lambda: hpack_ctx.hpack_encode_blocks(np.array([0, 1], np.uint64), np.zeros(8, np.uint8),
                                                       np.array([0, 6, 4], np.uint64), out_capacity=64)):
        with pytest.raises(pkg.CodecError) as err:
            call()
        assert err.value.code == pkg.capi.AWS_ERROR_INVALID_ARGUMENT


@pytest.mark.gpu
def test_device_pointer_round_trip_at_probe_scale(hpack_ctx):
    """256K header lists of 8-24 fields through the device entry points: encode, decode, and the lists come back."""
    import torch
    probe = _load("header_blocks_probe", "tools", "header_blocks_probe.py")
    dev = torch.device("cuda", 0)
    lists = probe.synthetic_lists(262_144, 1, dev)
    r = probe.round_trip(hpack_ctx, lists, dev)
    fo, strings, so, never = lists
    assert int(r["status"].abs().sum().item()) == 0
    assert torch.equal(r["field_offsets"], fo)
    F = int(fo[-1].item())
    assert torch.equal(r["string_offsets"][:2 * F + 1], so)
    assert torch.equal(r["strings"][:strings.numel()], strings)
    kinds = r["field_kind"][:F]
    assert bool((kinds[never.bool()] == NV).all())
