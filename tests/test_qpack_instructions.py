"""QPACK encoder- and decoder-stream instructions (RFC 9204 sections 4.3, 4.4;
include/aws/compression/qpack_instruction_batch.h).

CPU part (-m "not gpu"): the oracle (oracle/qpack_instruction_oracle.py) against RFC 9204 Appendix B's instruction
octets, which encode back to themselves; the appendix driven from octets alone (encoder-stream octets -> instruction
records -> a table kept here -> the section oracle -> the RFC's header lists); hand-built chunks of every kind and
every error rule; every appendix stream cut at every octet; the capacity bound; the header compiles and its struct
matches ctypes; no device means no result.
GPU part: every call through the C ABI against that oracle, array for array."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_qpack_field_sections import (HEADER_LISTS, RFC9204_SECTIONS, CallerTable, ROUTES, _any_bytes, _batch, _load,
                                       _routes, _text)

io = _load("qpack_instruction_oracle", "oracle", "qpack_instruction_oracle.py")
q = io.sections
lit = io.lit
ENC, DEC = io.ENCODER_STREAM, io.DECODER_STREAM
IS, ID, IL, DUP, CAP, ACK, CANCEL, ICI, AUTO = range(9)

# RFC 9204 Appendix B instruction octets: (stream, hex, [(kind, index, name, value)])
RFC9204_INSTRUCTIONS = [
    (ENC, "3fbd01", [(CAP, 220, b"", b"")]),                                                         # B.2
    (ENC, "c00f7777772e6578616d706c652e636f6d", [(IS, 0, b":authority", b"www.example.com")]),
    (ENC, "c10c2f73616d706c652f70617468", [(IS, 1, b":path", b"/sample/path")]),
    (ENC, "4a637573746f6d2d6b65790c637573746f6d2d76616c7565", [(IL, 0, b"custom-key", b"custom-value")]),  # B.3
    (ENC, "02", [(DUP, 2, b"", b"")]),                                                               # B.4
    (ENC, "810d637573746f6d2d76616c756532", [(ID, 1, b"", b"custom-value2")]),                       # B.5
    (DEC, "84", [(ACK, 4, b"", b"")]),                                                               # B.2
    (DEC, "01", [(ICI, 1, b"", b"")]),                                                               # B.3
    (DEC, "48", [(CANCEL, 8, b"", b"")]),                                                            # B.5
]
# the encoder-stream octets a decoder has read before each field section of RFC9204_SECTIONS
ENCODER_STREAM_OCTETS = {"B.1": "", "B.2": "3fbd01" "c00f7777772e6578616d706c652e636f6d" "c10c2f73616d706c652f70617468",
                         "B.4": "4a637573746f6d2d6b65790c637573746f6d2d76616c7565" "02"}


class InstructionTable(CallerTable):
    """The dynamic table of test_qpack_field_sections.py, fed decoded instruction records instead of parsed inserts."""

    def apply_records(self, records):
        for kind, index, name, value in records:
            if kind == CAP:
                self.max_entries = index // 32
            elif kind in (IS, IL):
                self.entries.append((name, value))
            elif kind == ID:
                self.entries.append((self.entries[len(self.entries) - 1 - index][0], value))
            elif kind == DUP:
                self.entries.append(self.entries[len(self.entries) - 1 - index])


@pytest.fixture(scope="module")
def instruction_oracle(oracle, oracle_tables):
    return io.InstructionOracle(lit.LiteralOracle(oracle, oracle_tables["hpack"]))


@pytest.fixture(scope="module")
def section_oracle(oracle, oracle_tables):
    return q.SectionOracle(lit.LiteralOracle(oracle, oracle_tables["hpack"]))


_HUFF = bytes.fromhex("f1e3c2e5f23a6ba0ab90f4ff")  # "www.example.com" (RFC 7541 C.4.1)


def _hand_vectors():
    """(stream, chunk, status, consumed, records): every kind, cuts, and one case per error rule."""
    long_name = b"n" * 40
    return [
        (ENC, b"\xc0\x00", lit.OK, 2, [(IS, 0, b":authority", b"")]),
        (ENC, b"\xff\x23\x01v", lit.OK, 4, [(IS, 98, b"x-frame-options", b"v")]),           # 6-bit prefix, 2 octets
        (ENC, b"\xe1\x00", lit.OK, 2, [(IS, 33, b"access-control-allow-headers", b"")]),
        (ENC, b"\x80\x01x", lit.OK, 3, [(ID, 0, b"", b"x")]),
        (ENC, b"\xbf\x81\x01\x00", lit.OK, 4, [(ID, 63 + 129, b"", b"")]),
        (ENC, b"\x41x\x00", lit.OK, 3, [(IL, 0, b"x", b"")]),                                  # raw name literal
        (ENC, b"\x5f\x09" + long_name + b"\x01v", lit.OK, 44, [(IL, 0, long_name, b"v")]),   # 5-bit length 31 + 9
        (ENC, b"\x6c" + _HUFF + b"\x8c" + _HUFF, lit.OK, 26, [(IL, 0, b"www.example.com", b"www.example.com")]),
        (ENC, b"\x00\x1f\x00", lit.OK, 3, [(DUP, 0, b"", b""), (DUP, 31, b"", b"")]),
        (ENC, b"\x20\x3f\xe1\x04", lit.OK, 4, [(CAP, 0, b"", b""), (CAP, 31 + 97 + 4 * 128, b"", b"")]),
        (DEC, b"\x80\xff\x00", lit.OK, 3, [(ACK, 0, b"", b""), (ACK, 127, b"", b"")]),
        (DEC, b"\x40\x7f\x01", lit.OK, 3, [(CANCEL, 0, b"", b""), (CANCEL, 64, b"", b"")]),
        (DEC, b"\x3f\x00", lit.OK, 2, [(ICI, 63, b"", b"")]),
        (ENC, b"", lit.OK, 0, []),
        (DEC, b"", lit.OK, 0, []),
        # cuts: the complete instructions are reported, the cut one is not
        (ENC, b"\x02\x3f", lit.OK, 1, [(DUP, 2, b"", b"")]),                                  # inside an integer
        (ENC, b"\xc1", lit.OK, 0, []),                                                        # before the value
        (ENC, b"\xc1\x05ab", lit.OK, 0, []),                                                  # inside the value
        (ENC, b"\x45ab", lit.OK, 0, []),                                                      # inside the name
        (ENC, b"\x43abc", lit.OK, 0, []),                                                     # a whole name, no value
        (ENC, b"\x61\xff", lit.OK, 0, []),                                                    # a bad name is not decoded
        (ENC, b"\x61\xff\x05ab", lit.OK, 0, []),                                              # ... when the value is cut
        (DEC, b"\x84\xff", lit.OK, 1, [(ACK, 4, b"", b"")]),
        (DEC, b"\x3f" + b"\xff" * 9, lit.OK, 0, []),                                          # nine continuations, cut
        # errors
        (ENC, b"\xff\x24\x00", lit.INVALID_ARGUMENT, 0, None),                                # static name index 99
        (ENC, b"\xff\x24", lit.INVALID_ARGUMENT, 0, None),                                    # ... read in full
        (ENC, b"\x02\xff\xe4\x00", lit.INVALID_ARGUMENT, 0, None),                            # after a good one
        (DEC, b"\x84\x00", lit.INVALID_ARGUMENT, 0, None),                                    # Insert Count Increment 0
        (DEC, b"\x7f" + b"\xff" * 9 + b"\x01", lit.INVALID_ARGUMENT, 0, None),                # an integer over 62 bits
        (ENC, b"\x1f" + b"\xff" * 9 + b"\x01", lit.INVALID_ARGUMENT, 0, None),
        (ENC, b"\x5f" + b"\xff" * 9 + b"\x01", lit.INVALID_ARGUMENT, 0, None),                # a name length
        (ENC, b"\xc1\x7f" + b"\xff" * 9 + b"\x01", lit.INVALID_ARGUMENT, 0, None),            # a value length
        (ENC, b"\x6d" + _HUFF + b"\xff\x00", lit.INVALID_PADDING, 0, None),                   # a whole octet of padding
        (ENC, b"\x70" + _HUFF + b"\xff" * 4 + b"\x00", lit.UNKNOWN_SYMBOL, 0, None),          # EOS in a name
        (ENC, b"\xc1\x81\xff", lit.INVALID_PADDING, 0, None),                                 # ... in a value
        (ENC, b"\xc1\x81\xff\xff\x24", lit.INVALID_PADDING, 0, None),                         # Huffman error first ...
        (ENC, b"\xff\x24\xc1\x81\xff", lit.INVALID_ARGUMENT, 0, None),                        # ... unless structure's is
        # a literal name that fails structurally after its name: the name's Huffman error comes first
        (ENC, b"\x61\xff\x7f" + b"\xff" * 9 + b"\x01", lit.INVALID_PADDING, 0, None),
        (ENC, b"\x41a\x7f" + b"\xff" * 9 + b"\x01", lit.INVALID_ARGUMENT, 0, None),           # a good name
    ]


# ------------------------------------------------------------------------------------------------ CPU
def test_oracle_decodes_rfc9204_appendix_b(instruction_oracle):
    for which, hexed, records in RFC9204_INSTRUCTIONS:
        data = bytes.fromhex(hexed)
        assert instruction_oracle.decode_chunk(which, data) == (lit.OK, len(data), records), hexed


def test_oracle_records_encode_back_to_the_rfc_bytes(instruction_oracle):
    for which, hexed, records in RFC9204_INSTRUCTIONS:
        data = b"".join(instruction_oracle.encode_instruction(which, k, i, n, v, lit.NEVER) for k, i, n, v in records)
        assert data == bytes.fromhex(hexed)
    assert instruction_oracle.encode_instruction(ENC, AUTO, 7, b":path", b"/sample/path", lit.NEVER) == \
        bytes.fromhex("c10c2f73616d706c652f70617468")                                   # AUTO: static name 1
    assert instruction_oracle.encode_instruction(ENC, AUTO, 7, b"custom-key", b"custom-value", lit.NEVER) == \
        bytes.fromhex("4a637573746f6d2d6b65790c637573746f6d2d76616c7565")               # AUTO: literal name


def test_rfc_chain_from_encoder_stream_octets(instruction_oracle, section_oracle):
    """Encoder-stream octets -> instruction records -> table -> section records -> the RFC's header lists, with no
    hand-parsed insert on the way; the last chunk is fed in pieces, its tail carried forward."""
    table = InstructionTable(capacity=0)
    want = {"B.1": (0, 0), "B.2": (2, 0), "B.4": (4, 4)}
    for name in ("B.1", "B.2", "B.4"):
        stream, tail = bytes.fromhex(ENCODER_STREAM_OCTETS[name]), b""
        for cut in range(0, len(stream) + 1, 5):
            chunk = tail + stream[cut:cut + 5]
            st, used, records = instruction_oracle.decode_chunk(ENC, chunk)
            assert st == lit.OK
            table.apply_records(records)
            tail = chunk[used:]
        assert tail == b""
        st, prefix, records = section_oracle.decode_section(bytes.fromhex(RFC9204_SECTIONS[name][0]))
        ric, base, headers = table.resolve(prefix, records)
        assert st == lit.OK and (ric, base) == want[name] and headers == HEADER_LISTS[name], name
    assert table.max_entries == 6 and table.size == 217


def test_oracle_hand_built_chunks(instruction_oracle):
    for which, chunk, status, consumed, records in _hand_vectors():
        st, used, got = instruction_oracle.decode_chunk(which, chunk)
        assert (st, used) == (status, consumed), chunk.hex()
        assert got == (records if status == lit.OK else []), chunk.hex()


def test_every_appendix_stream_cut_at_every_octet(instruction_oracle):
    for which in (ENC, DEC):
        items = [(bytes.fromhex(h), r) for w, h, r in RFC9204_INSTRUCTIONS if w == which]
        stream = b"".join(d for d, _ in items)
        ends = np.cumsum([len(d) for d, _ in items])
        for cut in range(len(stream) + 1):
            whole = int((ends <= cut).sum())
            st, used, got = instruction_oracle.decode_chunk(which, stream[:cut])
            assert st == lit.OK and used == (int(ends[whole - 1]) if whole else 0)
            assert got == [rec for _, r in items[:whole] for rec in r]


def test_capacity_bound_is_14_octets_per_input_octet():
    """The most string octets one input octet can yield: a two-octet insert with a one-octet static index (< 63) and
    an empty value, a three-octet one with a two-octet index, a name literal (one octet of Huffman: 8/5 symbols)."""
    one = max(len(n) for n, _ in q.STATIC_TABLE[:63]) / 2
    three = max(len(n) for n, _ in q.STATIC_TABLE[63:]) / 3
    assert one == 14 and q.STATIC_TABLE[33][0] == b"access-control-allow-headers"
    assert three < 14 and 8 / 5 < 14


def test_oracle_random_streams_round_trip(instruction_oracle):
    rng = np.random.default_rng(5)
    for which in (ENC, DEC):
        kinds = set()
        for mode in (lit.SMALLEST, lit.NEVER, lit.ALWAYS, None):
            data, records = instruction_oracle.random_stream(rng, which, _any_bytes, 200, mode)
            assert instruction_oracle.decode_chunk(which, data) == (lit.OK, len(data), records)
            kinds |= {r[0] for r in records}
            if mode is not None:
                again = b"".join(instruction_oracle.encode_instruction(which, k, i, n, v, mode) for k, i, n, v in records)
                assert again == data
        assert kinds == set(io.STREAM_KINDS[which])


def test_header_compiles_as_c_and_cxx(pkg, tmp_path):
    inc = [a for d in pkg._build.INCLUDES for a in ("-I", d)]
    for compiler, ext, std in (("gcc", "c", "-std=c99"), ("g++", "cpp", "-std=c++14")):
        src = tmp_path / ("instructions." + ext)
        src.write_text("#include <aws/compression/qpack_instruction_batch.h>\n"
                       "int main(void){struct aws_qpack_instructions s; enum aws_qpack_instruction_kind k = "
                       "AWS_QPACK_INSERT_AUTO; enum aws_qpack_instruction_stream w = AWS_QPACK_DECODER_STREAM; "
                       "(void)s; (void)k; (void)w; return 0;}\n")
        subprocess.check_call([compiler, std, "-Wall", "-Werror", *inc, "-c", "-o", str(tmp_path / "o.o"), str(src)])


def test_instructions_struct_matches_the_header(pkg, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <aws/compression/qpack_instruction_batch.h>\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %d %d\\n", sizeof(struct aws_qpack_instructions),'
                   'offsetof(struct aws_qpack_instructions, instruction_capacity),'
                   'offsetof(struct aws_qpack_instructions, strings),'
                   'offsetof(struct aws_qpack_instructions, string_offsets), sizeof(enum aws_qpack_instruction_kind),'
                   '(int)AWS_QPACK_INSERT_AUTO, (int)AWS_QPACK_DECODER_STREAM);return 0;}\n')
    exe = tmp_path / "layout"
    inc = [a for d in pkg._build.INCLUDES for a in ("-I", d)]
    subprocess.check_call(["gcc", "-std=gnu99", *inc, "-o", str(exe), str(src)])
    t = pkg.capi.aws_qpack_instructions
    assert subprocess.check_output([str(exe)], text=True).split() == [
        str(C.sizeof(t)), str(t.instruction_capacity.offset), str(t.strings.offset), str(t.string_offsets.offset),
        str(C.sizeof(C.c_int)), str(pkg.capi.QPACK_INSERT_AUTO), str(pkg.capi.QPACK_DECODER_STREAM)]


def test_no_device_means_no_result(pkg, coders, product):
    """Without a device there is no context, and without a context every instruction entry point fails with
    AWS_ERROR_INVALID_ARGUMENT, writing nothing, instead of computing anything on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.CodecError) as err:
        pkg.BatchContext(coders.coder("hpack"), device=0)
    assert err.value.code == pkg.AWS_ERROR_COMPRESSION_DEVICE_FAILURE
    L = product.lib
    data = np.frombuffer(bytes.fromhex("c00f7777772e6578616d706c652e636f6d"), np.uint8)
    offs = np.array([0, len(data)], np.uint64)
    io_, so, idx, consumed = (np.full(k, 7, np.uint64) for k in (2, 3, 1, 1))
    kind, strings = np.full(1, 7, np.uint8), np.full(32, 7, np.uint8)
    instr = pkg.capi.aws_qpack_instructions(1, io_.ctypes.data, 1, kind.ctypes.data, idx.ctypes.data,
                                            strings.ctypes.data, 32, so.ctypes.data)
    out = np.zeros(8, np.uint8)
    status = np.full(1, 7, np.int32)
    S = C.byref(instr)
    calls = [
        lambda: L.aws_qpack_instruction_decode_batch(None, ENC, 1, data.ctypes.data, offs.ctypes.data, S,
                                                     consumed.ctypes.data, status.ctypes.data),
        lambda: L.aws_qpack_instruction_encode_batch(None, ENC, S, 0, out.ctypes.data, 8, offs.ctypes.data,
                                                     status.ctypes.data),
        lambda: L.aws_qpack_instruction_decode_batch_device(None, DEC, 1, data.ctypes.data, offs.ctypes.data,
                                                            len(data), S, consumed.ctypes.data, status.ctypes.data, None),
        lambda: L.aws_qpack_instruction_encode_batch_device(None, ENC, S, 1, 0, 0, out.ctypes.data, 8,
                                                            offs.ctypes.data, status.ctypes.data, None),
    ]
    for call in calls:
        L.aws_reset_error()
        assert call() == pkg.capi.AWS_OP_ERR
        assert L.aws_last_error() == pkg.capi.AWS_ERROR_INVALID_ARGUMENT
    for a in (io_, so, idx, consumed, kind, strings, status):
        assert (a == 7).all()
    assert not out.any() and list(offs) == [0, len(data)]


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def hpack_ctx(pkg, coders):
    ctx = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
    yield ctx
    ctx.close()


def assert_decode_matches(got, want):
    assert np.array_equal(got["status"], want["status"]), np.flatnonzero(got["status"] != want["status"])[:10]
    assert np.array_equal(got["consumed"], want["consumed"]), np.flatnonzero(got["consumed"] != want["consumed"])[:10]
    assert np.array_equal(got["instruction_offsets"], want["instruction_offsets"])
    ni = int(want["instruction_offsets"][-1])
    for name in ("kind", "index"):
        assert np.array_equal(got[name][:ni], want[name]), name
    assert np.array_equal(got["string_offsets"][:2 * ni + 1], want["string_offsets"])
    assert np.array_equal(got["strings"][:len(want["strings"])], want["strings"])


def _random_chunks(instruction_oracle, rng, which, n, make_string=_any_bytes, mode=None, cut=True):
    """n chunks of random instructions; with cut, most chunks end at a random octet (inside an instruction or not)."""
    chunks = []
    for _ in range(n):
        data, _ = instruction_oracle.random_stream(rng, which, make_string, int(rng.integers(0, 12)), mode)
        if cut and data and rng.random() < 0.7:
            data = data[:int(rng.integers(0, len(data) + 1))]
        chunks.append(data)
    return chunks


@pytest.mark.gpu
def test_appendix_b_instructions_in_one_batch(hpack_ctx, instruction_oracle):
    for which in (ENC, DEC):
        chunks = [bytes.fromhex(h) for w, h, _ in RFC9204_INSTRUCTIONS if w == which]
        data, offs = _batch(chunks)
        want = instruction_oracle.decode_batch(which, data, offs)
        got = hpack_ctx.qpack_decode_instructions(which, data, offs)
        assert_decode_matches(got, want)
        assert not want["status"].any() and np.array_equal(want["consumed"], np.diff(offs))
        n = int(want["instruction_offsets"][-1])
        enc = hpack_ctx.qpack_encode_instructions(which, want["instruction_offsets"], want["kind"], want["index"],
                                                  want["strings"], want["string_offsets"][:2 * n + 1], 256,
                                                  mode=lit.NEVER)
        assert not enc["status"].any() and bytes(enc["out"][:int(enc["out_offsets"][-1])]) == bytes(data)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES)
def test_random_chunks_match_oracle(hpack_ctx, instruction_oracle, monkeypatch, pkg, coders, route):
    ctx = _routes(monkeypatch, pkg, coders, route) or hpack_ctx
    rng = np.random.default_rng(31)
    for which in (ENC, DEC):
        chunks = _random_chunks(instruction_oracle, rng, which, 2000) + [b"", b"\x02"]
        rng.shuffle(chunks)
        data, offs = _batch(chunks)
        want = instruction_oracle.decode_batch(which, data, offs)
        assert_decode_matches(ctx.qpack_decode_instructions(which, data, offs), want)
        assert set(want["kind"]) == set(io.STREAM_KINDS[which]) and not want["status"].any()
        assert (want["consumed"] < np.diff(offs)).any()


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES)
def test_malformed_chunks_report_the_first_error_and_nothing_else(hpack_ctx, instruction_oracle, monkeypatch, pkg,
                                                                  coders, route):
    ctx = _routes(monkeypatch, pkg, coders, route) or hpack_ctx
    cases = _hand_vectors()
    for which in (ENC, DEC):
        chunks = [c for w, c, _, _, _ in cases if w == which] * 3
        data, offs = _batch(chunks)
        want = instruction_oracle.decode_batch(which, data, offs)
        got = ctx.qpack_decode_instructions(which, data, offs)
        assert_decode_matches(got, want)
        bad = got["status"] != 0
        assert bad.any() and not got["consumed"][bad].any()
        assert (np.diff(got["instruction_offsets"].astype(np.int64))[bad] == 0).all()
    # a batch whose only literal belongs to no instruction
    alone = ctx.qpack_decode_instructions(ENC, np.frombuffer(b"\x61\xff\x7f" + b"\xff" * 9 + b"\x01", np.uint8),
                                          np.array([0, 13], np.uint64))
    assert list(alone["status"]) == [lit.INVALID_PADDING] and list(alone["instruction_offsets"]) == [0, 0]


def _records(want):
    n = int(want["instruction_offsets"][-1])
    return want["instruction_offsets"], want["kind"][:n], want["index"][:n], want["strings"], \
        want["string_offsets"][:2 * n + 1]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.SMALLEST, lit.NEVER, lit.ALWAYS])
def test_encode_matches_oracle_and_decodes_back(hpack_ctx, instruction_oracle, mode):
    rng = np.random.default_rng(60 + mode)
    for which in (ENC, DEC):
        chunks = _random_chunks(instruction_oracle, rng, which, 800, _text, cut=False)
        want = instruction_oracle.decode_batch(which, *_batch(chunks))
        io_, kind, index, strings, so = _records(want)
        kind = kind.copy()
        if which == ENC:
            kind[np.flatnonzero((kind == IS) | (kind == IL))[::2]] = AUTO        # the name match chooses
        data, offs, status = instruction_oracle.encode_batch(which, io_, kind, index, strings, so, mode)
        assert not status.any()
        got = hpack_ctx.qpack_encode_instructions(which, io_, kind, index, strings, so, len(data) + 64, mode=mode)
        assert not got["status"].any() and np.array_equal(got["out_offsets"], offs)
        assert np.array_equal(got["out"][:len(data)], data)
        back = hpack_ctx.qpack_decode_instructions(which, data, offs)
        assert not back["status"].any() and np.array_equal(back["consumed"], np.diff(offs))
        assert np.array_equal(back["instruction_offsets"], io_)
        assert np.array_equal(back["string_offsets"][:len(so)], so) and np.array_equal(back["strings"][:len(strings)],
                                                                                      strings)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.NEVER, lit.ALWAYS])
def test_decode_records_encode_gives_back_the_consumed_octets(hpack_ctx, instruction_oracle, mode):
    rng = np.random.default_rng(80 + mode)
    for which in (ENC, DEC):
        chunks = _random_chunks(instruction_oracle, rng, which, 1500, mode=mode)
        data, offs = _batch(chunks)
        got = hpack_ctx.qpack_decode_instructions(which, data, offs)
        assert not got["status"].any()
        io_, kind, index, strings, so = _records(got)
        enc = hpack_ctx.qpack_encode_instructions(which, io_, kind, index, strings[:int(so[-1])], so, len(data) + 64,
                                                  mode=mode)
        assert not enc["status"].any() and np.array_equal(np.diff(enc["out_offsets"]), got["consumed"])
        want = b"".join(c[:int(u)] for c, u in zip(chunks, got["consumed"]))
        assert bytes(enc["out"][:len(want)]) == want


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.SMALLEST, lit.ALWAYS])
def test_invalid_chunks_among_valid_ones(hpack_ctx, instruction_oracle, mode):
    rng = np.random.default_rng(95 + mode)
    for which in (ENC, DEC):
        chunks = _random_chunks(instruction_oracle, rng, which, 300, _text, cut=False)
        want = instruction_oracle.decode_batch(which, *_batch(chunks))
        io_, kind, index, strings, so = [a.copy() for a in _records(want)]
        n = len(io_) - 1
        damage = []
        for b in rng.choice(n, size=60, replace=False):
            f0, f1 = int(io_[b]), int(io_[b + 1])
            if f1 == f0:
                continue
            how = int(rng.integers(0, 5))
            if how == 0:
                kind[f0] = 9                                            # a kind above AUTO
            elif how == 1:
                kind[f0] = ACK if which == ENC else IS                  # a kind of the other stream
            elif how == 2:
                kind[f0], index[f0] = (IS, 99) if which == ENC else (ICI, 0)
            elif how == 3:
                kind[f0], index[f0] = (DUP if which == ENC else ACK), (1 << 64) - 1  # an integer a decoder refuses
            else:
                kind[f0] = AUTO if which == DEC else 10                 # AUTO on the decoder stream
            damage.append(b)
        data, offs, status = instruction_oracle.encode_batch(which, io_, kind, index, strings, so, mode)
        assert (status[damage] == lit.INVALID_ARGUMENT).all() and (status == 0).sum() >= n - 60
        got = hpack_ctx.qpack_encode_instructions(which, io_, kind, index, strings, so, len(data) + 64, mode=mode)
        assert np.array_equal(got["status"], status)
        assert np.array_equal(got["out_offsets"], offs) and np.array_equal(got["out"][:len(data)], data)


@pytest.mark.gpu
def test_empty_batches_and_empty_chunks(hpack_ctx, instruction_oracle):
    for which in (ENC, DEC):
        empty = hpack_ctx.qpack_decode_instructions(which, np.zeros(0, np.uint8), np.zeros(1, np.uint64))
        assert list(empty["instruction_offsets"]) == [0] and list(empty["string_offsets"][:1]) == [0]
        none = hpack_ctx.qpack_decode_instructions(which, np.zeros(0, np.uint8), np.zeros(4, np.uint64))
        assert list(none["instruction_offsets"]) == [0] * 4 and not none["consumed"].any() and not none["status"].any()
        enc = hpack_ctx.qpack_encode_instructions(which, np.zeros(1, np.uint64), np.zeros(0, np.uint8),
                                                  np.zeros(0, np.uint64), np.zeros(0, np.uint8), np.zeros(1, np.uint64), 8)
        assert list(enc["out_offsets"]) == [0]
        enc = hpack_ctx.qpack_encode_instructions(which, np.zeros(4, np.uint64), np.zeros(0, np.uint8),
                                                  np.zeros(0, np.uint64), np.zeros(0, np.uint8), np.zeros(1, np.uint64), 8)
        assert list(enc["out_offsets"]) == [0] * 4 and not enc["status"].any()
    # empty chunks between others
    chunks = [b"", bytes.fromhex("c10c2f73616d706c652f70617468"), b"", b"\x02\x3f", b""]
    data, offs = _batch(chunks)
    assert_decode_matches(hpack_ctx.qpack_decode_instructions(ENC, data, offs),
                          instruction_oracle.decode_batch(ENC, data, offs))


@pytest.mark.gpu
def test_capacity_contract(hpack_ctx, instruction_oracle, pkg):
    rng = np.random.default_rng(4)
    chunks = _random_chunks(instruction_oracle, rng, ENC, 200, _text)
    data, offs = _batch(chunks)
    want = instruction_oracle.decode_batch(ENC, data, offs)
    ni, ns = int(want["instruction_offsets"][-1]), len(want["strings"])
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.qpack_decode_instructions(ENC, data, offs, instruction_capacity=ni - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    for name in ("instruction_offsets", "consumed", "status"):
        assert np.array_equal(err.value.result[name], want[name]), name
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.qpack_decode_instructions(ENC, data, offs, instruction_capacity=ni, strings_capacity=ns - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    assert np.array_equal(err.value.result["string_offsets"], want["string_offsets"])
    assert_decode_matches(hpack_ctx.qpack_decode_instructions(ENC, data, offs, instruction_capacity=ni,
                                                              strings_capacity=ns), want)
    # the documented bounds hold on the worst chunk: every insert two octets of 28 string octets
    worst = np.frombuffer(b"\xe1\x00" * 2048, np.uint8)
    got = hpack_ctx.qpack_decode_instructions(ENC, worst, np.array([0, len(worst)], np.uint64))
    assert int(got["instruction_offsets"][-1]) == 2048 and int(got["string_offsets"][2 * 2048]) == 14 * len(worst)
    # the decoder stream needs no strings at all
    acks = np.frombuffer(b"\x84\x01\x48" * 100, np.uint8)
    dec = hpack_ctx.qpack_decode_instructions(DEC, acks, np.array([0, len(acks)], np.uint64), strings_capacity=0)
    assert int(dec["instruction_offsets"][-1]) == 300 and not dec["string_offsets"].any()
    io_, kind, index, strings, so = _records(want)
    enc = hpack_ctx.qpack_encode_instructions(ENC, io_, kind, index, strings, so, 1 << 20)
    total = int(enc["out_offsets"][-1])
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.qpack_encode_instructions(ENC, io_, kind, index, strings, so, total - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    assert np.array_equal(err.value.result["out_offsets"], enc["out_offsets"])
    assert np.array_equal(err.value.result["status"], enc["status"])
    exact = hpack_ctx.qpack_encode_instructions(ENC, io_, kind, index, strings, so, total)
    assert np.array_equal(exact["out"][:total], enc["out"][:total])
    # decreasing offsets, encode offsets that do not start at 0, and a stream other than 0 or 1 are refused
    for call in (lambda: hpack_ctx.qpack_decode_instructions(ENC, data, np.array([0, 5, 2, len(data)], np.uint64)),
                 lambda: hpack_ctx.qpack_decode_instructions(2, data, offs),
                 lambda: hpack_ctx.qpack_encode_instructions(ENC, np.array([1, 2], np.uint64), np.zeros(2, np.uint8),
                                                             np.zeros(2, np.uint64), np.zeros(8, np.uint8),
                                                             np.array([0, 2, 4, 6, 8], np.uint64), 64),
                 lambda: hpack_ctx.qpack_encode_instructions(ENC, io_, kind, index, strings, so, 64, mode=3)):
        with pytest.raises(pkg.CodecError) as err:
            call()
        assert err.value.code == pkg.capi.AWS_ERROR_INVALID_ARGUMENT


@pytest.mark.gpu
def test_device_calls_on_a_caller_stream_at_unaligned_addresses(hpack_ctx, instruction_oracle):
    """The _device forms with every array in its own allocation at an odd phase behind guard bytes (the helpers of
    test_gpu_device_calls.py), on a caller stream: results equal the oracle's, nothing is written past a capacity or
    a guard, and the inputs are unchanged."""
    import torch
    from test_gpu_device_calls import place, scratch_array

    rng = np.random.default_rng(34)
    st = torch.cuda.Stream(torch.device("cuda", 0))
    with torch.cuda.stream(st):
        for which in (ENC, DEC):
            chunks = _random_chunks(instruction_oracle, rng, which, 400, _text, mode=lit.SMALLEST) + [b""]
            data, offs = _batch(chunks)
            want = instruction_oracle.decode_batch(which, data, offs)
            n, ni, ns = len(chunks), int(want["instruction_offsets"][-1]), len(want["strings"])
            d_in, d_off = place(data, 3, "echo"), place(offs, 8)
            arrays = {"instruction_offsets": scratch_array(np.uint64, n + 1, 8), "kind": scratch_array(np.uint8, ni, 5),
                      "index": scratch_array(np.uint64, ni, 8), "string_offsets": scratch_array(np.uint64, 2 * ni + 1, 8),
                      "consumed": scratch_array(np.uint64, n, 8), "status": scratch_array(np.int32, n, 4)}
            if which == ENC:
                arrays["strings"] = scratch_array(np.uint8, ns, 7)
            a = arrays
            hpack_ctx.qpack_decode_instructions_device(
                which, n, d_in, d_off, len(data), a["instruction_offsets"], a["kind"], a["index"], a.get("strings"),
                a["string_offsets"], a["consumed"], status=a["status"], stream=st.cuda_stream, instruction_capacity=ni,
                strings_capacity=ns)
            st.synchronize()
            got = {k: v.read(k) for k, v in arrays.items()}
            got.setdefault("strings", np.zeros(0, np.uint8))
            d_in.read("in", unchanged=True)
            d_off.read("in_offsets", unchanged=True)
            assert_decode_matches(got, want)
            # encode the records into an output of exactly the consumed size
            io_, kind, index, strings, so = _records(want)
            expect = b"".join(c[:int(u)] for c, u in zip(chunks, want["consumed"]))
            expect_offs = np.concatenate([[0], np.cumsum(want["consumed"])]).astype(np.uint64)
            i = {"io": place(io_, 8), "kind": place(kind, 7), "index": place(index, 8)}
            if which == ENC:
                i.update(strings=place(strings, 5, "ones"), so=place(so, 8))
            out, out_offs = scratch_array(np.uint8, len(expect), 9), scratch_array(np.uint64, n + 1, 8)
            status = scratch_array(np.int32, n, 4)
            hpack_ctx.qpack_encode_instructions_device(
                which, n, i["io"], ni, i["kind"], i["index"], i.get("strings"), i.get("so"),
                ns if which == ENC else 0, out, out_offs, status=status, mode=lit.SMALLEST, out_capacity=len(expect),
                stream=st.cuda_stream)
            st.synchronize()
            assert np.array_equal(out_offs.read("out_offsets"), expect_offs)
            assert bytes(out.read("out")) == expect
            assert not status.read("status").any()
            for name, arr in i.items():
                arr.read(name, unchanged=True)


@pytest.mark.gpu
def test_full_rfc_chain_on_the_gpu(hpack_ctx):
    """Appendix B end to end through the device: the encoder stream in pieces (tails carried forward), the inserts
    applied to the table, the sections decoded, and the acknowledgments and increments encoded on the decoder stream."""
    table = InstructionTable(capacity=0)
    want = {"B.1": (0, 0), "B.2": (2, 0), "B.4": (4, 4)}
    acks = []
    for name in ("B.1", "B.2", "B.4"):
        stream, tail = bytes.fromhex(ENCODER_STREAM_OCTETS[name]), b""
        for cut in range(0, len(stream) + 1, 7):
            chunk = np.frombuffer(tail + stream[cut:cut + 7], np.uint8)
            got = hpack_ctx.qpack_decode_instructions(ENC, chunk, np.array([0, len(chunk)], np.uint64))
            assert not got["status"].any()
            n = int(got["instruction_offsets"][-1])
            so, s = got["string_offsets"], got["strings"]
            table.apply_records([(int(got["kind"][f]), int(got["index"][f]), bytes(s[int(so[2 * f]):int(so[2 * f + 1])]),
                                  bytes(s[int(so[2 * f + 1]):int(so[2 * f + 2])])) for f in range(n)])
            tail = bytes(chunk[int(got["consumed"][0]):])
        assert tail == b""
        section = np.frombuffer(bytes.fromhex(RFC9204_SECTIONS[name][0]), np.uint8)
        dec = hpack_ctx.qpack_decode_sections(section, np.array([0, len(section)], np.uint64))
        nf = int(dec["field_offsets"][-1])
        so, s = dec["string_offsets"], dec["strings"]
        records = [(int(dec["field_kind"][f]), int(dec["field_index"][f]), int(dec["never_indexed"][f]),
                    bytes(s[int(so[2 * f]):int(so[2 * f + 1])]), bytes(s[int(so[2 * f + 1]):int(so[2 * f + 2])]))
                   for f in range(nf)]
        prefix = tuple(int(dec[k][0]) for k in ("encoded_insert_count", "base_sign", "delta_base"))
        ric, base, headers = table.resolve(prefix, records)
        assert (ric, base) == want[name] and headers == HEADER_LISTS[name], name
        if ric:
            acks.append(ric)
    # the decoder acknowledges the two sections that referenced the table (streams 4 and 8 in the appendix) and
    # raises the Known Received Count past the insert that no section has referenced yet
    enc = hpack_ctx.qpack_encode_instructions(DEC, np.array([0, 1, 2, 3], np.uint64), np.array([ACK, ICI, CANCEL], np.uint8),
                                              np.array([4, 1, 8], np.uint64), np.zeros(0, np.uint8), np.zeros(7, np.uint64),
                                              16)
    assert acks == [2, 4] and not enc["status"].any()
    assert bytes(enc["out"][:3]) == bytes.fromhex("840148") and list(enc["out_offsets"]) == [0, 1, 2, 3]


@pytest.mark.gpu
def test_device_pointer_round_trip_at_probe_scale(hpack_ctx):
    """The probe's workload (256K encoder-stream chunks, about 4M instructions, and a decoder-stream chunk per
    connection) through the device entry points: encode, decode, and the records come back."""
    import torch
    probe = _load("qpack_instructions_probe", "tools", "qpack_instructions_probe.py")
    dev = torch.device("cuda", 0)
    for which, batch in zip((ENC, DEC), probe.synthetic_streams(262_144, 1, dev)):
        kinds = probe._check(probe.round_trip(hpack_ctx, which, batch, dev), batch)
        assert all(kinds[k] for k in io.STREAM_KINDS[which] if k != ID)
