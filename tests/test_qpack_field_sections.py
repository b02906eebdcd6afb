"""QPACK field sections (RFC 9204 section 4.5, Appendix A; include/aws/compression/qpack_field_section_batch.h).

CPU part (-m "not gpu"): the static table of the device code against the oracle's own transcription
(oracle/qpack_field_section_oracle.py); the oracle against RFC 9204 Appendix B: every section decodes to the RFC's
field lines, and a dynamic table kept here (fed the appendix's encoder-stream inserts as data) rebuilds the RFC's
header lists from the prefix and the records alone; the records encode back to the RFC's bytes; hand-built vectors
for every line kind and every error rule; the capacity bound; the stateless encoder rules; the header compiles; no
device means no result.
GPU part: every call through the C ABI against that oracle, array for array."""
import ctypes as C
import importlib.util
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(name, *path):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, *path))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module


q = _load("qpack_field_section_oracle", "oracle", "qpack_field_section_oracle.py")
lit = q.lit
IS, ID, IPB, NRS, NRD, NRPB, LN, AUTO = range(8)

# RFC 9204 Appendix B field sections: (hex, (encoded insert count, S, Delta Base), [(kind, index, N, value)])
RFC9204_SECTIONS = {
    "B.1": ("0000510b2f696e6465782e68746d6c", (0, 0, 0), [(NRS, 1, 0, b"/index.html")]),
    "B.2": ("03811011", (3, 1, 1), [(IPB, 0, 0, b""), (IPB, 1, 0, b"")]),
    "B.4": ("050080c181", (5, 0, 0), [(ID, 0, 0, b""), (IS, 1, 0, b""), (ID, 1, 0, b"")]),
}
# The encoder-stream instructions before each section (RFC 9204 B.2 - B.4), as the caller's table sees them:
# ("insert", name, value) or ("duplicate", relative index).
ENCODER_STREAM = {
    "B.1": [],
    "B.2": [("insert", b":authority", b"www.example.com"), ("insert", b":path", b"/sample/path")],
    "B.4": [("insert", b"custom-key", b"custom-value"), ("duplicate", 2)],  # (B.3's insert, then B.4's duplicate)
}
HEADER_LISTS = {
    "B.1": [(b":path", b"/index.html")],
    "B.2": [(b":authority", b"www.example.com"), (b":path", b"/sample/path")],
    "B.4": [(b":authority", b"www.example.com"), (b":path", b"/"), (b"custom-key", b"custom-value")],
}


def expected_records(lines):
    return [(k, i, n) + q.field_strings(k, i, b"", v) for k, i, n, v in lines]


class CallerTable:
    """A decoder's dynamic table (RFC 9204 3.2) with the section-prefix arithmetic of 4.5.1, driven by the encoder
    stream's inserts and by the decoder's prefix and records alone. Capacity 220: MaxEntries = 220 // 32 = 6."""

    def __init__(self, capacity=220):
        self.max_entries = capacity // 32
        self.entries = []  # absolute index -> (name, value)

    def apply(self, instructions):
        for op in instructions:
            if op[0] == "insert":
                self.entries.append(op[1:])
            else:
                self.entries.append(self.entries[len(self.entries) - 1 - op[1]])

    @property
    def size(self):
        return sum(32 + len(n) + len(v) for n, v in self.entries)

    def required_insert_count(self, encoded):
        if encoded == 0:
            return 0
        full_range = 2 * self.max_entries
        assert encoded <= full_range
        max_value = len(self.entries) + self.max_entries
        max_wrapped = (max_value // full_range) * full_range
        ric = max_wrapped + encoded - 1
        if ric > max_value:
            assert ric > full_range
            ric -= full_range
        assert ric != 0
        return ric

    def resolve(self, prefix, records):
        ric = self.required_insert_count(prefix[0])
        base = ric - prefix[2] - 1 if prefix[1] else ric + prefix[2]
        headers = []
        for kind, index, _, name, value in records:
            if kind in (ID, NRD):
                absolute = base - 1 - index
            elif kind in (IPB, NRPB):
                absolute = base + index
            else:
                headers.append((name, value))
                continue
            assert absolute < ric
            entry = self.entries[absolute]
            headers.append(entry if kind in (ID, IPB) else (entry[0], value))
        return ric, base, headers


@pytest.fixture(scope="module")
def section_oracle(oracle, oracle_tables):
    return q.SectionOracle(lit.LiteralOracle(oracle, oracle_tables["hpack"]))


def _text(rng, length):
    return bytes(rng.choice(np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789-_/:;=, ", np.uint8), size=length))


def _any_bytes(rng, length):
    return rng.integers(0, 256, size=length, dtype=np.uint8).tobytes() if rng.random() < 0.2 else _text(rng, length)


def _batch(items):
    offs = np.zeros(len(items) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(b) for b in items])
    return np.frombuffer(b"".join(items), dtype=np.uint8), offs


def _random_lists(rng, n, max_fields=10, empty_sections=0.05):
    """Header lists mixing exact static entries, static names and custom names (empty strings too)."""
    names = [n for n, _ in q.STATIC_TABLE] + [b"x-custom", b"custom-key", b"", b"X-Upper"]
    fields, never = [], []
    offs = [0]
    for _ in range(n):
        count = 0 if rng.random() < empty_sections else int(rng.integers(0, max_fields + 1))
        for _ in range(count):
            r = rng.random()
            if r < 0.25:
                fields += list(q.STATIC_TABLE[int(rng.integers(0, 99))])
            else:
                fields += [names[int(rng.integers(0, len(names)))] if r < 0.8 else _text(rng, int(rng.integers(1, 20))),
                           _any_bytes(rng, int(rng.choice([0, 3, 17, 60, 130])))]
            never.append(1 if rng.random() < 0.15 else 0)
        offs.append(len(never))
    string_offsets = np.zeros(len(fields) + 1, dtype=np.uint64)
    string_offsets[1:] = np.cumsum([len(s) for s in fields])
    return (np.array(offs, dtype=np.uint64), np.frombuffer(b"".join(fields), dtype=np.uint8), string_offsets,
            np.array(never, dtype=np.uint8))


# ------------------------------------------------------------------------------------------------ CPU
def test_device_static_table_is_the_oracles():
    """Two transcriptions of Appendix A agree: the blob and offsets of qpack_sections.cuh, and the oracle's table."""
    src = open(os.path.join(ROOT, "aws-c-compression_b200", "csrc", "qpack_sections.cuh")).read()
    blob_src = re.search(r"kQpackStaticBlob\[\] =(.*?);\s*static_assert", src, re.S).group(1)
    blob = "".join(re.findall(r'"((?:[^"\\]|\\.)*)"', blob_src)).encode()
    offs = [int(x) for x in re.search(r"kQpackStaticOff\[[^\]]*\] = \{(.*?)\}", src, re.S).group(1).split(",")]
    assert blob == b"".join(n + v for n, v in q.STATIC_TABLE) and len(blob) == 2026
    assert len(offs) == 2 * 99 + 1
    assert [(blob[offs[2 * i]:offs[2 * i + 1]], blob[offs[2 * i + 1]:offs[2 * i + 2]]) for i in range(99)] == q.STATIC_TABLE


def test_capacity_bound_is_69_octets_per_input_octet():
    """The most string octets one input octet can yield: one-octet INDEXED_STATIC lines (index < 63), two-octet
    ones, and a one-octet NAME_REF_STATIC (index < 15) with the shortest value literal; Huffman gives 8/5."""
    one = max(len(n) + len(v) for n, v in q.STATIC_TABLE[:63])
    two = max(len(n) + len(v) for n, v in q.STATIC_TABLE[63:]) / 2
    name_ref = max(len(n) for n, _ in q.STATIC_TABLE[:15]) / 2
    assert one == 69 and q.STATIC_TABLE[58] == (b"strict-transport-security",
                                                b"max-age=31536000; includesubdomains; preload")
    assert two < 69 and name_ref < 69 and 8 / 5 < 69


def test_oracle_decodes_rfc9204_appendix_b(section_oracle):
    for name, (hexed, prefix, lines) in RFC9204_SECTIONS.items():
        assert section_oracle.decode_section(bytes.fromhex(hexed)) == (lit.OK, prefix, expected_records(lines)), name


def test_prefix_and_records_are_enough_to_rebuild_the_rfc_header_lists(section_oracle):
    """B.1 (RIC 0, Base 0), B.2 (encoded 3: RIC 2, S = 1, Delta Base 1: Base 0), B.4 (encoded 5: RIC 4, Base 4; the
    duplicated :authority is absolute 3). RFC 9204 B.5 has no field section (an insert and a stream cancellation)."""
    table = CallerTable()
    want = {"B.1": (0, 0), "B.2": (2, 0), "B.4": (4, 4)}
    for name in ("B.1", "B.2", "B.4"):
        table.apply(ENCODER_STREAM[name])
        st, prefix, records = section_oracle.decode_section(bytes.fromhex(RFC9204_SECTIONS[name][0]))
        assert st == lit.OK
        ric, base, headers = table.resolve(prefix, records)
        assert (ric, base) == want[name] and headers == HEADER_LISTS[name], name
    assert table.size == 217  # (the table size the RFC shows after B.4)


def _records_of(section_oracle, sections):
    want = section_oracle.decode_batch(*_batch(sections))
    return want, (want["encoded_insert_count"], want["base_sign"], want["delta_base"], want["field_offsets"],
                  want["field_kind"], want["field_index"], want["strings"], want["string_offsets"], want["never_indexed"])


def test_oracle_records_encode_back_to_the_rfc_bytes(section_oracle):
    sections = [bytes.fromhex(h) for h, _, _ in RFC9204_SECTIONS.values()]
    _, r = _records_of(section_oracle, sections)
    data, offs, status = section_oracle.encode_records_batch(*r[:8], never_indexed=r[8], mode=lit.NEVER)
    assert not status.any() and bytes(data) == b"".join(sections)


_HUFF = bytes.fromhex("f1e3c2e5f23a6ba0ab90f4ff")  # "www.example.com" (RFC 7541 C.4.1)


def _hand_vectors():
    """(section, status, records): every line kind, and one case per error rule, behind a valid prefix."""
    v = [
        (b"\x00\x00\xc0", lit.OK, [(IS, 0, 0) + q.STATIC_TABLE[0]]),
        (b"\x00\x00\xfa", lit.OK, [(IS, 58, 0) + q.STATIC_TABLE[58]]),
        (b"\x00\x00\xff\x23\xe2", lit.OK, [(IS, 98, 0) + q.STATIC_TABLE[98], (IS, 34, 0) + q.STATIC_TABLE[34]]),
        (b"\x02\x00\x8a", lit.OK, [(ID, 10, 0, b"", b"")]),
        (b"\x02\x00\xbf\x81\x01", lit.OK, [(ID, 63 + 129, 0, b"", b"")]),          # 6-bit prefix, 3 octets
        (b"\x02\x00\x1f\x00", lit.OK, [(IPB, 15, 0, b"", b"")]),                     # post-base, 4-bit prefix full
        (b"\x00\x00\x72\x01a", lit.OK, [(NRS, 2, 1, b"age", b"a")]),                   # static name, N = 1
        (b"\x00\x00\x5f\x00\x00", lit.OK, [(NRS, 15, 0, b":method", b"")]),          # 4-bit prefix full
        (b"\x02\x00\x6f\x0a\x01x", lit.OK, [(NRD, 25, 1, b"", b"x")]),                # relative name, N = 1
        (b"\x02\x00\x0f\x0a\x01x", lit.OK, [(NRPB, 17, 1, b"", b"x")]),               # post-base name, N = 1
        (b"\x02\x00\x02\x00", lit.OK, [(NRPB, 2, 0, b"", b"")]),
        (b"\x00\x00\x21x\x00", lit.OK, [(LN, 0, 0, b"x", b"")]),                      # raw name literal
        (b"\x00\x00\x37\x00" + b"abcdefg" + b"\x01v", lit.OK, [(LN, 0, 1, b"abcdefg", b"v")]),  # 3-bit length 7, N
        (b"\x00\x00\x2f\x05" + _HUFF + b"\x00", lit.OK, [(LN, 0, 0, b"www.example.com", b"")]),  # Huffman name
        (b"\x00\x00\x51\x8c" + _HUFF, lit.OK, [(NRS, 1, 0, b":path", b"www.example.com")]),  # Huffman value
        (b"\xff\x01\xff\x7f", lit.OK, []),                                           # 2-octet prefix integers, no lines
        (b"\x00\x80", lit.OK, []),                                                   # S = 1, Delta Base 0
        # errors
        (b"", lit.SHORT_BUFFER, None),                                               # an empty item
        (b"\x00", lit.SHORT_BUFFER, None),                                           # cut inside the prefix
        (b"\xff", lit.SHORT_BUFFER, None),                                           # ... inside its first integer
        (b"\x00\x7f", lit.SHORT_BUFFER, None),                                       # ... inside Delta Base
        (b"\x00\x00\xff", lit.SHORT_BUFFER, None),                                   # cut inside an index
        (b"\x00\x00\x51\x05ab", lit.SHORT_BUFFER, None),                             # cut inside a value literal
        (b"\x00\x00\x51", lit.SHORT_BUFFER, None),                                   # no value literal
        (b"\x00\x00\x23ab", lit.SHORT_BUFFER, None),                                 # cut inside a name literal
        (b"\x00\x00\xff\x24", lit.INVALID_ARGUMENT, None),                           # static index 99
        (b"\x00\x00\x5f\x54\x00", lit.INVALID_ARGUMENT, None),                       # static name index 99
        (b"\x00\x00\x80", lit.INVALID_ARGUMENT, None),                               # dynamic line, RIC 0
        (b"\x00\x00\x10", lit.INVALID_ARGUMENT, None),                               # post-base line, RIC 0
        (b"\x00\x00\x40\x00", lit.INVALID_ARGUMENT, None),                           # dynamic name, RIC 0
        (b"\x00\x00\x00\x00", lit.INVALID_ARGUMENT, None),                           # post-base name, RIC 0
        (b"\x00\x00\xbf", lit.INVALID_ARGUMENT, None),                               # ... refused at its first octet
        (b"\xff" + b"\xff" * 9 + b"\x01\x00", lit.INVALID_ARGUMENT, None),           # a prefix integer over 62 bits
        (b"\x02\x00\xbf" + b"\xff" * 9 + b"\x01", lit.INVALID_ARGUMENT, None),       # an index over 62 bits
        (b"\x00\x00\x27" + b"\xff" * 9 + b"\x01", lit.INVALID_ARGUMENT, None),       # a name length over 62 bits
        (b"\x00\x00\x2f\x06" + _HUFF + b"\xff\x00", lit.INVALID_PADDING, None),     # a whole octet of padding
        (b"\x00\x00\x2f\x09" + _HUFF + b"\xff" * 4 + b"\x00", lit.UNKNOWN_SYMBOL, None),  # EOS in a name
        (b"\x00\x00\x51\x81\xff", lit.INVALID_PADDING, None),                         # ... in a value literal
        (b"\x00\x00\x51\x90" + _HUFF + b"\xff" * 4, lit.UNKNOWN_SYMBOL, None),
        (b"\x00\x00\x51\x81\xff\xff\x24", lit.INVALID_PADDING, None),                 # Huffman error first ...
        (b"\x00\x00\xff\x24\x51\x81\xff", lit.INVALID_ARGUMENT, None),                # ... unless structure's is
        # a literal name that fails after its name: the name's Huffman error comes first
        (b"\x00\x00\x29\xff", lit.INVALID_PADDING, None),                            # bad name, no value literal
        (b"\x00\x00\x29\xff\x05", lit.INVALID_PADDING, None),                        # bad name, value cut short
        (b"\x00\x00\x29\xff\x7f" + b"\xff" * 9 + b"\x01", lit.INVALID_PADDING, None),  # value length over 62 bits
        (b"\x00\x00\x21a\x05", lit.SHORT_BUFFER, None),                              # a good name, value cut short
        (b"\x00\x00\xc1\x29\xff\xc1", lit.INVALID_PADDING, None),
        (b"\x00\x00\xff\x24\x29\xff", lit.INVALID_ARGUMENT, None),                   # the structural error first
    ]
    return v


def test_oracle_hand_built_sections(section_oracle):
    for section, status, records in _hand_vectors():
        st, prefix, got = section_oracle.decode_section(section)
        assert st == status, section.hex()
        if status == lit.OK:
            assert got == records, section.hex()
        else:
            assert got == [] and prefix == (0, 0, 0)


def test_oracle_stateless_encoder_rules(section_oracle):
    enc = section_oracle.encode_field
    assert enc(b":path", b"/") == bytes.fromhex("c1")                                  # exact static match
    assert enc(b":path", b"/index.html", mode=lit.NEVER) == bytes.fromhex(RFC9204_SECTIONS["B.1"][0])[2:]
    assert enc(b":path", b"/", True, lit.NEVER) == bytes.fromhex("7101") + b"/"           # never-indexed beats exact
    assert enc(b"x-secret", b"s", True, lit.NEVER) == b"\x37\x01x-secret\x01s"         # literal name, N = 1, 3-bit len 7+1
    assert enc(b"custom", b"v", mode=lit.NEVER) == b"\x26custom\x01v"
    assert enc(b":status", b"302") == bytes.fromhex("ff03")                              # index 66: two octets
    assert enc(b":status", b"201", mode=lit.NEVER) == bytes.fromhex("5f09") + b"\x03201"  # lowest :status index 24
    assert enc(b"x-frame-options", b"sameorigin") == bytes.fromhex("ff23")              # index 98: two octets
    assert enc(b":authority", b"") == bytes.fromhex("c0")                               # index 0, empty value
    huff = enc(b"x-custom-name", b"", mode=lit.ALWAYS)
    assert huff[0] & 0xF8 == 0x28 and section_oracle.decode_section(b"\x00\x00" + huff)[2] == [
        (LN, 0, 0, b"x-custom-name", b"")]
    data, offs = section_oracle.encode_batch(np.array([0, 0, 1], np.uint64), np.frombuffer(b":path/", np.uint8),
                                             np.array([0, 5, 6], np.uint64))
    assert bytes(data) == bytes.fromhex("0000" "0000c1") and list(offs) == [0, 2, 5]   # an empty list: its prefix


def test_oracle_encode_then_decode_is_the_identity(section_oracle):
    rng = np.random.default_rng(3)
    fo, strings, so, never = _random_lists(rng, 60)
    for mode in (lit.SMALLEST, lit.NEVER, lit.ALWAYS):
        data, offs = section_oracle.encode_batch(fo, strings, so, never, mode)
        got = section_oracle.decode_batch(data, offs)
        assert not got["status"].any() and np.array_equal(got["field_offsets"], fo)
        assert np.array_equal(got["string_offsets"], so) and np.array_equal(got["strings"], strings)
        assert np.array_equal(got["never_indexed"], never)
        assert set(got["field_kind"]) <= {IS, NRS, LN} and IS not in set(got["field_kind"][never == 1])


def test_random_writer_emits_every_kind_and_its_records(section_oracle):
    rng = np.random.default_rng(8)
    kinds, nevers, widths = set(), set(), set()
    for _ in range(400):
        section, prefix, records = section_oracle.random_section(rng, _any_bytes)
        assert section_oracle.decode_section(section) == (lit.OK, prefix, records)
        kinds |= {r[0] for r in records}
        nevers |= {r[2] for r in records}
        widths |= {("eic", prefix[0] >= 255), ("delta", prefix[2] >= 127)}
        widths |= {("name", len(r[3]) >= 7) for r in records if r[0] == LN}
    assert kinds == set(range(7)) and nevers == {0, 1}
    assert {("eic", True), ("delta", True), ("name", True)} <= widths


def test_header_compiles_as_c_and_cxx(pkg, tmp_path):
    inc = [a for d in pkg._build.INCLUDES for a in ("-I", d)]
    for compiler, ext, std in (("gcc", "c", "-std=c99"), ("g++", "cpp", "-std=c++14")):
        src = tmp_path / ("sections." + ext)
        src.write_text("#include <aws/compression/qpack_field_section_batch.h>\n"
                       "int main(void){struct aws_qpack_field_sections s; enum aws_qpack_field_kind k = "
                       "AWS_QPACK_FIELD_LITERAL_NAME; (void)s; (void)k; return 0;}\n")
        subprocess.check_call([compiler, std, "-Wall", "-Werror", *inc, "-c", "-o", str(tmp_path / "o.o"), str(src)])


def test_sections_struct_matches_the_header(pkg, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <aws/compression/qpack_field_section_batch.h>\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void){printf("%zu %zu %zu %zu %d\\n", sizeof(struct aws_qpack_field_sections),'
                   'offsetof(struct aws_qpack_field_sections, field_offsets),'
                   'offsetof(struct aws_qpack_field_sections, never_indexed),'
                   'offsetof(struct aws_qpack_field_sections, string_offsets), (int)AWS_QPACK_FIELD_AUTO);return 0;}\n')
    exe = tmp_path / "layout"
    inc = [a for d in pkg._build.INCLUDES for a in ("-I", d)]
    subprocess.check_call(["gcc", "-std=gnu99", *inc, "-o", str(exe), str(src)])
    t = pkg.capi.aws_qpack_field_sections
    assert subprocess.check_output([str(exe)], text=True).split() == [
        str(C.sizeof(t)), str(t.field_offsets.offset), str(t.never_indexed.offset), str(t.string_offsets.offset),
        str(pkg.capi.QPACK_FIELD_AUTO)]


def test_no_device_means_no_result(pkg, coders, product):
    """Without a device there is no context (AWS_ERROR_COMPRESSION_DEVICE_FAILURE), and without a context every
    field-section entry point fails with AWS_ERROR_INVALID_ARGUMENT, writing nothing, instead of computing anything on
    the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.CodecError) as err:
        pkg.BatchContext(coders.coder("hpack"), device=0)
    assert err.value.code == pkg.AWS_ERROR_COMPRESSION_DEVICE_FAILURE
    L = product.lib
    data = np.frombuffer(bytes.fromhex("0000c1"), np.uint8)
    offs = np.array([0, 3], np.uint64)
    eic, delta, fo, so, idx = (np.full(k, 7, np.uint64) for k in (1, 1, 2, 3, 1))
    sign, kind, never = (np.full(1, 7, np.uint8) for _ in range(3))
    sections = pkg.capi.aws_qpack_field_sections(1, eic.ctypes.data, sign.ctypes.data, delta.ctypes.data, fo.ctypes.data,
                                                 1, kind.ctypes.data, idx.ctypes.data, never.ctypes.data, None, 0,
                                                 so.ctypes.data)
    out = np.zeros(8, np.uint8)
    status = np.full(1, 7, np.int32)
    S = C.byref(sections)
    calls = [
        lambda: L.aws_qpack_field_section_decode_batch(None, 1, data.ctypes.data, offs.ctypes.data, S, status.ctypes.data),
        lambda: L.aws_qpack_field_section_encode_batch(None, S, 0, out.ctypes.data, 8, offs.ctypes.data),
        lambda: L.aws_qpack_field_section_encode_records_batch(None, S, 0, out.ctypes.data, 8, offs.ctypes.data,
                                                               status.ctypes.data),
        lambda: L.aws_qpack_field_section_decode_batch_device(None, 1, data.ctypes.data, offs.ctypes.data, 3, S,
                                                              status.ctypes.data, None),
        lambda: L.aws_qpack_field_section_encode_batch_device(None, S, 1, 0, 0, out.ctypes.data, 8, offs.ctypes.data,
                                                              None),
        lambda: L.aws_qpack_field_section_encode_records_batch_device(None, S, 1, 0, 0, out.ctypes.data, 8,
                                                                      offs.ctypes.data, status.ctypes.data, None),
    ]
    for call in calls:
        L.aws_reset_error()
        assert call() == pkg.capi.AWS_OP_ERR
        assert L.aws_last_error() == pkg.capi.AWS_ERROR_INVALID_ARGUMENT
    for a in (eic, delta, fo, so, idx, sign, kind, never, status):
        assert (a == 7).all()
    assert not out.any() and list(offs) == [0, 3]


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def hpack_ctx(pkg, coders):
    ctx = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
    yield ctx
    ctx.close()


DECODE_ARRAYS = ("encoded_insert_count", "base_sign", "delta_base")


def assert_decode_matches(got, want):
    assert np.array_equal(got["status"], want["status"]), np.flatnonzero(got["status"] != want["status"])[:10]
    for name in DECODE_ARRAYS + ("field_offsets",):
        assert np.array_equal(got[name], want[name]), name
    nf = int(want["field_offsets"][-1])
    for name in ("field_kind", "field_index", "never_indexed"):
        assert np.array_equal(got[name][:nf], want[name]), name
    assert np.array_equal(got["string_offsets"][:2 * nf + 1], want["string_offsets"])
    assert np.array_equal(got["strings"][:len(want["strings"])], want["strings"])


def _routes(monkeypatch, pkg, coders, route):
    """The context and environment of one literal route."""
    if route == "passes":
        monkeypatch.setenv("AWS_HUFFMAN_HPACK_PASSES", "1")
    if route == "generic":
        monkeypatch.setenv("AWS_HUFFMAN_BATCH_FORCE_GENERIC", "1")
        ctx = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
        monkeypatch.delenv("AWS_HUFFMAN_BATCH_FORCE_GENERIC")
        return ctx
    return None


ROUTES = ["one_kernel", "passes", "generic"]


@pytest.mark.gpu
def test_appendix_b_sections_in_one_batch(hpack_ctx, section_oracle):
    sections = [bytes.fromhex(h) for h, _, _ in RFC9204_SECTIONS.values()]
    data, offs = _batch(sections)
    want = section_oracle.decode_batch(data, offs)
    assert_decode_matches(hpack_ctx.qpack_decode_sections(data, offs), want)
    assert not want["status"].any() and list(want["encoded_insert_count"]) == [0, 3, 5]
    records = (want["encoded_insert_count"], want["base_sign"], want["delta_base"], want["field_kind"], want["field_index"])
    enc = hpack_ctx.qpack_encode_sections(want["field_offsets"], want["strings"], want["string_offsets"], 64,
                                          mode=lit.NEVER, never_indexed=want["never_indexed"], records=records)
    assert not enc["status"].any() and bytes(enc["out"][:int(enc["out_offsets"][-1])]) == bytes(data)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES)
def test_random_sections_match_oracle(hpack_ctx, section_oracle, monkeypatch, pkg, coders, route):
    ctx = _routes(monkeypatch, pkg, coders, route) or hpack_ctx
    rng = np.random.default_rng(21)
    sections = [section_oracle.random_section(rng, _any_bytes)[0] for _ in range(2500)] + [b"\x00\x00", b"\x05\x81"]
    rng.shuffle(sections)
    data, offs = _batch(sections)
    want = section_oracle.decode_batch(data, offs)
    assert_decode_matches(ctx.qpack_decode_sections(data, offs), want)
    assert set(want["field_kind"]) == set(range(7)) and not want["status"].any()


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES)
def test_malformed_sections_report_the_first_error_and_nothing_else(hpack_ctx, section_oracle, monkeypatch, pkg, coders,
                                                                    route):
    ctx = _routes(monkeypatch, pkg, coders, route) or hpack_ctx
    cases = _hand_vectors()
    sections = [s for s, _, _ in cases] * 3
    data, offs = _batch(sections)
    want = section_oracle.decode_batch(data, offs)
    assert list(want["status"][:len(cases)]) == [st for _, st, _ in cases]
    got = ctx.qpack_decode_sections(data, offs)
    assert_decode_matches(got, want)
    bad = got["status"] != 0
    assert (np.diff(got["field_offsets"].astype(np.int64))[bad] == 0).all()
    assert not got["encoded_insert_count"][bad].any() and not got["delta_base"][bad].any()
    # a batch whose only literal belongs to no field
    alone = ctx.qpack_decode_sections(np.frombuffer(b"\x00\x00\x29\xff", np.uint8), np.array([0, 4], np.uint64))
    assert list(alone["status"]) == [lit.INVALID_PADDING] and list(alone["field_offsets"]) == [0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.SMALLEST, lit.NEVER, lit.ALWAYS])
def test_encode_matches_oracle_and_decodes_back(hpack_ctx, section_oracle, mode):
    rng = np.random.default_rng(50 + mode)
    fo, strings, so, never = _random_lists(rng, 800)
    want, want_offs = section_oracle.encode_batch(fo, strings, so, never, mode)
    got = hpack_ctx.qpack_encode_sections(fo, strings, so, out_capacity=len(want) + 64, mode=mode, never_indexed=never)
    assert np.array_equal(got["out_offsets"], want_offs)
    assert np.array_equal(got["out"][:len(want)], want)
    back = hpack_ctx.qpack_decode_sections(want, want_offs)
    assert not back["status"].any() and np.array_equal(back["field_offsets"], fo)
    assert np.array_equal(back["string_offsets"][:len(so)], so) and np.array_equal(back["strings"][:len(strings)], strings)
    kinds = back["field_kind"][:len(never)]
    assert np.array_equal(back["never_indexed"][:len(never)], never)
    assert set(kinds) == {IS, NRS, LN} and not (kinds[never == 1] == IS).any()
    assert not back["encoded_insert_count"].any() and not back["delta_base"].any()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.NEVER, lit.ALWAYS])
def test_decode_records_encode_gives_back_the_sections(hpack_ctx, section_oracle, mode):
    rng = np.random.default_rng(70 + mode)
    sections = [section_oracle.random_section(rng, _any_bytes, mode=mode)[0] for _ in range(1500)] + [b"\x00\x00"]
    data, offs = _batch(sections)
    got = hpack_ctx.qpack_decode_sections(data, offs)
    assert not got["status"].any()
    F = int(got["field_offsets"][-1])
    records = tuple(got[k] for k in DECODE_ARRAYS) + (got["field_kind"][:F], got["field_index"][:F])
    S = int(got["string_offsets"][2 * F])
    enc = hpack_ctx.qpack_encode_sections(got["field_offsets"], got["strings"][:S], got["string_offsets"][:2 * F + 1],
                                          len(data) + 64, mode=mode, never_indexed=got["never_indexed"][:F],
                                          records=records)
    assert not enc["status"].any() and np.array_equal(enc["out_offsets"], offs)
    assert np.array_equal(enc["out"][:len(data)], data)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.SMALLEST, lit.ALWAYS])
def test_records_encode_with_invalid_sections_among_valid_ones(hpack_ctx, section_oracle, mode):
    rng = np.random.default_rng(90 + mode)
    sections = [section_oracle.random_section(rng, _text)[0] for _ in range(300)]
    _, r = _records_of(section_oracle, sections)
    eic, sign, delta, fo, kind, index, strings, so, never = [a.copy() for a in r]
    kind[::7] = AUTO                                          # the stateless rules for some fields
    n = len(fo) - 1
    damage = []
    for b in rng.choice(n, size=60, replace=False):
        f0, f1 = int(fo[b]), int(fo[b + 1])
        how = int(rng.integers(0, 6)) if f1 > f0 else int(rng.integers(3, 5))
        if how == 0:
            kind[f0] = 8                                      # a kind above AUTO
        elif how == 1:
            kind[f0], index[f0] = IS, 99                       # static index 99
        elif how == 2:
            kind[f0], index[f0] = NRS, 1000
        elif how == 3:
            sign[b] = 2                                       # S neither 0 nor 1
        elif how == 4:
            eic[b] = (1 << 64) - 1                            # a prefix integer a decoder refuses
        else:
            eic[b] = 0                                        # a dynamic reference with RIC 0
            kind[f0], index[f0] = IPB, 0
        damage.append(b)
    want, want_offs, want_status = section_oracle.encode_records_batch(eic, sign, delta, fo, kind, index, strings, so,
                                                                       never, mode)
    assert (want_status[damage] == lit.INVALID_ARGUMENT).all()
    got = hpack_ctx.qpack_encode_sections(fo, strings, so, len(want) + 64, mode=mode, never_indexed=never,
                                          records=(eic, sign, delta, kind, index))
    assert np.array_equal(got["status"], want_status)
    assert np.array_equal(got["out_offsets"], want_offs) and np.array_equal(got["out"][:len(want)], want)
    # an index a decoder refuses (over 9 continuation octets), a name index at the 4-bit limit's edge
    one = hpack_ctx.qpack_encode_sections(np.array([0, 1, 2], np.uint64), np.zeros(0, np.uint8), np.zeros(5, np.uint64),
                                          64, records=(np.array([2, 2], np.uint64), np.zeros(2, np.uint8),
                                                       np.zeros(2, np.uint64), np.array([ID, ID], np.uint8),
                                                       np.array([(1 << 64) - 1, (1 << 63) + 62], np.uint64)))
    assert list(one["status"]) == [lit.INVALID_ARGUMENT, lit.OK]


@pytest.mark.gpu
def test_capacity_contract(hpack_ctx, section_oracle, pkg):
    rng = np.random.default_rng(4)
    sections = [section_oracle.random_section(rng, _text)[0] for _ in range(200)]
    data, offs = _batch(sections)
    want = section_oracle.decode_batch(data, offs)
    nf, ns = int(want["field_offsets"][-1]), len(want["strings"])
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.qpack_decode_sections(data, offs, field_capacity=nf - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    for name in DECODE_ARRAYS + ("field_offsets", "status"):
        assert np.array_equal(err.value.result[name], want[name]), name
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.qpack_decode_sections(data, offs, field_capacity=nf, strings_capacity=ns - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    assert np.array_equal(err.value.result["field_offsets"], want["field_offsets"])
    assert np.array_equal(err.value.result["string_offsets"], want["string_offsets"])
    assert_decode_matches(hpack_ctx.qpack_decode_sections(data, offs, field_capacity=nf, strings_capacity=ns), want)
    # the documented bounds hold on the worst section: every line one octet of 69 string octets
    worst = np.frombuffer(b"\x00\x00" + b"\xfa" * 4096, np.uint8)
    got = hpack_ctx.qpack_decode_sections(worst, np.array([0, len(worst)], np.uint64))
    assert int(got["field_offsets"][-1]) == 4096 and int(got["string_offsets"][2 * 4096]) == 69 * 4096
    enc = hpack_ctx.qpack_encode_sections(want["field_offsets"], want["strings"], want["string_offsets"], 1 << 20)
    total = int(enc["out_offsets"][-1])
    with pytest.raises(pkg.CodecError) as err:
        hpack_ctx.qpack_encode_sections(want["field_offsets"], want["strings"], want["string_offsets"], total - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    assert np.array_equal(err.value.result["out_offsets"], enc["out_offsets"])
    exact = hpack_ctx.qpack_encode_sections(want["field_offsets"], want["strings"], want["string_offsets"], total)
    assert np.array_equal(exact["out"][:total], enc["out"][:total])
    # decreasing offsets, and encode offsets that do not start at 0, are refused before any kernel reads them
    for call in (lambda: hpack_ctx.qpack_decode_sections(data, np.array([0, 5, 2, len(data)], np.uint64)),
                 lambda: hpack_ctx.qpack_encode_sections(np.array([1, 2], np.uint64), np.zeros(8, np.uint8),
                                                         np.array([0, 2, 4, 6, 8], np.uint64), 64),
                 lambda: hpack_ctx.qpack_encode_sections(np.array([0, 1], np.uint64), np.zeros(8, np.uint8),
                                                         np.array([2, 4, 6], np.uint64), 64)):
        with pytest.raises(pkg.CodecError) as err:
            call()
        assert err.value.code == pkg.capi.AWS_ERROR_INVALID_ARGUMENT


@pytest.mark.gpu
def test_empty_batches_and_sections_without_fields(hpack_ctx, section_oracle):
    empty = hpack_ctx.qpack_decode_sections(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    assert list(empty["field_offsets"]) == [0] and list(empty["string_offsets"][:1]) == [0]
    enc = hpack_ctx.qpack_encode_sections(np.zeros(1, np.uint64), np.zeros(0, np.uint8), np.zeros(1, np.uint64), 8)
    assert list(enc["out_offsets"]) == [0]
    # lists without fields are still sections (their prefix), stateless and from records alike
    fo = np.zeros(4, np.uint64)
    enc = hpack_ctx.qpack_encode_sections(fo, np.zeros(0, np.uint8), np.zeros(1, np.uint64), 8)
    assert list(enc["out_offsets"]) == [0, 2, 4, 6] and not enc["out"][:6].any()
    rec = hpack_ctx.qpack_encode_sections(fo, np.zeros(0, np.uint8), np.zeros(1, np.uint64), 16,
                                          records=(np.array([0, 300, 1], np.uint64), np.array([0, 1, 2], np.uint8),
                                                   np.array([0, 127, 0], np.uint64), np.zeros(0, np.uint8),
                                                   np.zeros(0, np.uint64)))
    assert list(rec["status"]) == [0, 0, lit.INVALID_ARGUMENT] and list(rec["out_offsets"]) == [0, 2, 6, 6]
    assert bytes(rec["out"][:6]) == b"\x00\x00\xff\x2d\xff\x00"
    # prefix-only sections between others, decoded
    sections = [b"\x00\x00", bytes.fromhex("0000c1"), b"\x07\x85", b"\x00\x00", bytes.fromhex("0000510b2f696e6465782e68746d6c")]
    data, offs = _batch(sections)
    assert_decode_matches(hpack_ctx.qpack_decode_sections(data, offs), section_oracle.decode_batch(data, offs))


@pytest.mark.gpu
def test_device_calls_on_a_caller_stream_at_unaligned_addresses(hpack_ctx, section_oracle, pkg):
    """The _device forms with every array in its own allocation at an odd phase behind guard bytes (the helpers of
    test_gpu_device_calls.py), on a caller stream: results equal the oracle's, nothing is written past a capacity or
    a guard, and the inputs are unchanged."""
    import torch
    from test_gpu_device_calls import place, scratch_array

    rng = np.random.default_rng(33)
    sections = [section_oracle.random_section(rng, _text, mode=lit.SMALLEST)[0] for _ in range(400)] + [b"\x00\x00"]
    data, offs = _batch(sections)
    want = section_oracle.decode_batch(data, offs)
    n, nf, ns = len(sections), int(want["field_offsets"][-1]), len(want["strings"])
    st = torch.cuda.Stream(torch.device("cuda", 0))
    with torch.cuda.stream(st):
        d_in, d_off = place(data, 3, "echo"), place(offs, 8)
        arrays = {"encoded_insert_count": scratch_array(np.uint64, n, 8), "base_sign": scratch_array(np.uint8, n, 1),
                  "delta_base": scratch_array(np.uint64, n, 8), "field_offsets": scratch_array(np.uint64, n + 1, 8),
                  "field_kind": scratch_array(np.uint8, nf, 5), "field_index": scratch_array(np.uint64, nf, 8),
                  "never_indexed": scratch_array(np.uint8, nf, 3), "strings": scratch_array(np.uint8, ns, 7),
                  "string_offsets": scratch_array(np.uint64, 2 * nf + 1, 8), "status": scratch_array(np.int32, n, 4)}
        a = arrays
        hpack_ctx.qpack_decode_sections_device(n, d_in, d_off, len(data), a["encoded_insert_count"], a["base_sign"],
                                               a["delta_base"], a["field_offsets"], a["field_kind"], a["field_index"],
                                               a["never_indexed"], a["strings"], a["string_offsets"], status=a["status"],
                                               stream=st.cuda_stream, field_capacity=nf, strings_capacity=ns)
        st.synchronize()
        got = {k: v.read(k) for k, v in arrays.items()}
        d_in.read("in", unchanged=True)
        d_off.read("in_offsets", unchanged=True)
        assert_decode_matches(got, want)
        # encode (stateless and records) into an output of exactly the size needed
        fo, strings, so, never = want["field_offsets"], want["strings"], want["string_offsets"], want["never_indexed"]
        plain, plain_offs = section_oracle.encode_batch(fo, strings, so, never)
        inputs = {"fo": place(fo, 8), "strings": place(strings, 5, "ones"), "so": place(so, 8), "never": place(never, 1),
                  "eic": place(want["encoded_insert_count"], 8), "sign": place(want["base_sign"], 3),
                  "delta": place(want["delta_base"], 8), "kind": place(want["field_kind"], 7),
                  "index": place(want["field_index"], 8)}
        i = inputs
        for records, expect, expect_offs in ((None, plain, plain_offs), ("records", data, offs)):
            out, out_offs = scratch_array(np.uint8, len(expect), 9), scratch_array(np.uint64, n + 1, 8)
            status = scratch_array(np.int32, n, 4)
            rec = (i["eic"], i["sign"], i["delta"], i["kind"], i["index"]) if records else None
            hpack_ctx.qpack_encode_sections_device(n, i["fo"], nf, i["strings"], i["so"], ns, out, out_offs,
                                                   mode=lit.SMALLEST, never_indexed=i["never"], records=rec,
                                                   status=status if records else None, out_capacity=len(expect),
                                                   stream=st.cuda_stream)
            st.synchronize()
            assert np.array_equal(out_offs.read("out_offsets"), expect_offs)
            assert np.array_equal(out.read("out"), expect)
            if records:
                assert not status.read("status").any()
        for name, arr in i.items():
            arr.read(name, unchanged=True)


@pytest.mark.gpu
def test_device_pointer_round_trip_at_probe_scale(hpack_ctx):
    """256K header lists of 8-24 fields through the device entry points: encode, decode, and the lists come back."""
    import torch
    probe = _load("qpack_sections_probe", "tools", "qpack_sections_probe.py")
    dev = torch.device("cuda", 0)
    lists = probe.synthetic_lists(262_144, 1, dev)
    r = probe.round_trip(hpack_ctx, lists, dev)
    fo, strings, so, never = lists
    assert int(r["status"].abs().sum().item()) == 0
    assert torch.equal(r["field_offsets"], fo)
    F = int(fo[-1].item())
    assert torch.equal(r["string_offsets"][:2 * F + 1], so)
    assert torch.equal(r["strings"][:strings.numel()], strings)
    assert torch.equal(r["never_indexed"][:F], never)
