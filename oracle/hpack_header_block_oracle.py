"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

CPU restatement of HPACK header blocks (RFC 7541 section 6 field representations over the section 5 primitives,
the Appendix A static table), built over the literal oracle (oracle/hpack_literals_oracle.py), used only as the
checker by tests/test_hpack_header_blocks.py.

Parity status: unpinned against the reference — the reference repository (awslabs/aws-c-compression) holds no
header-block code (its caller, aws-c-http, does). Pinned on RFC 7541 instead: the header blocks of Appendix C.2 to
C.6 decode to the RFC's representations and, through a dynamic table kept by the test, to the RFC's header lists.

It holds:
  * STATIC_TABLE (Appendix A);
  * BlockOracle.decode_block / decode_batch: the decode semantics of aws_hpack_header_block_decode_batch (one
    record per representation, static references resolved, dynamic references reported with empty strings, the
    first error a front-to-back decoder meets, zero fields for a failing block);
  * BlockOracle.encode_field / encode_batch: the stateless encoder's rules (never-indexed, exact static match, static
    name, literal name);
  * BlockOracle.random_block: a writer that emits every representation kind (the encoder never emits INCREMENTAL or
    size updates), with the records a decoder must return.

Pure-Python loops: fine for the test sizes.
"""
import importlib.util
import os

import numpy as np

_spec = importlib.util.spec_from_file_location(
    "hpack_literals_oracle", os.path.join(os.path.dirname(os.path.abspath(__file__)), "hpack_literals_oracle.py"))
lit = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(lit)

OK, SHORT_BUFFER, INVALID_ARGUMENT = lit.OK, lit.SHORT_BUFFER, lit.INVALID_ARGUMENT
INDEXED, INCREMENTAL, WITHOUT, NEVER, SIZE_UPDATE = range(5)
_PREFIX = {INDEXED: (7, 0x80), INCREMENTAL: (6, 0x40), WITHOUT: (4, 0x00), NEVER: (4, 0x10), SIZE_UPDATE: (5, 0x20)}

STATIC_TABLE = [(n.encode(), v.encode()) for n, v in [
    (":authority", ""), (":method", "GET"), (":method", "POST"), (":path", "/"), (":path", "/index.html"),
    (":scheme", "http"), (":scheme", "https"), (":status", "200"), (":status", "204"), (":status", "206"),
    (":status", "304"), (":status", "400"), (":status", "404"), (":status", "500"), ("accept-charset", ""),
    ("accept-encoding", "gzip, deflate"), ("accept-language", ""), ("accept-ranges", ""), ("accept", ""),
    ("access-control-allow-origin", ""), ("age", ""), ("allow", ""), ("authorization", ""), ("cache-control", ""),
    ("content-disposition", ""), ("content-encoding", ""), ("content-language", ""), ("content-length", ""),
    ("content-location", ""), ("content-range", ""), ("content-type", ""), ("cookie", ""), ("date", ""),
    ("etag", ""), ("expect", ""), ("expires", ""), ("from", ""), ("host", ""), ("if-match", ""),
    ("if-modified-since", ""), ("if-none-match", ""), ("if-range", ""), ("if-unmodified-since", ""),
    ("last-modified", ""), ("link", ""), ("location", ""), ("max-forwards", ""), ("proxy-authenticate", ""),
    ("proxy-authorization", ""), ("range", ""), ("referer", ""), ("refresh", ""), ("retry-after", ""),
    ("server", ""), ("set-cookie", ""), ("strict-transport-security", ""), ("transfer-encoding", ""),
    ("user-agent", ""), ("vary", ""), ("via", ""), ("www-authenticate", "")]]
assert len(STATIC_TABLE) == 61


def static_name_index(name):
    """The lowest Appendix A index whose name is `name`, or 0."""
    for i, (n, _) in enumerate(STATIC_TABLE):
        if n == name:
            return i + 1
    return 0


def static_exact_index(name, value):
    for i, entry in enumerate(STATIC_TABLE):
        if entry == (name, value):
            return i + 1
    return 0


def field_strings(kind, index, name=b"", value=b""):
    """The (name, value) a record carries: static references resolved, dynamic ones (>= 62) empty."""
    if kind == SIZE_UPDATE:
        return b"", b""
    if kind == INDEXED:
        return STATIC_TABLE[index - 1] if 1 <= index <= 61 else (b"", b"")
    if 1 <= index <= 61:
        name = STATIC_TABLE[index - 1][0]
    elif index > 61:
        name = b""
    return name, value


class BlockOracle:
    def __init__(self, literal_oracle):
        self.lit = literal_oracle

    # ---- decode ----
    def _literal(self, block, pos):
        """(status, string, new pos) for the string literal at block[pos:]."""
        if pos >= len(block):
            return SHORT_BUFFER, b"", pos
        length, used = lit.decode_integer(block[pos:], 7)
        if length is None:
            return used, b"", pos
        if length > len(block) - pos - used:
            return SHORT_BUFFER, b"", pos
        end = pos + used + length
        st, s = self.lit.decode(block[pos:end])
        return st, s, end

    def decode_block(self, block):
        """Returns (status, records) with records = [(kind, index, name, value)]; no records when status != OK."""
        block = bytes(block)
        pos, seen_field, records = 0, False, []
        while pos < len(block):
            b0 = block[pos]
            if b0 & 0x80:
                kind = INDEXED
            elif b0 & 0xE0 == 0x20:
                kind = SIZE_UPDATE
                if seen_field:
                    return INVALID_ARGUMENT, []
            else:
                kind = INCREMENTAL if b0 & 0x40 else (NEVER if b0 & 0x10 else WITHOUT)
            index, used = lit.decode_integer(block[pos:], _PREFIX[kind][0])
            if index is None:
                return used, []
            pos += used
            name = value = b""
            if kind == INDEXED and index == 0:
                return INVALID_ARGUMENT, []
            if kind in (INCREMENTAL, WITHOUT, NEVER):
                if index == 0:
                    st, name, pos = self._literal(block, pos)
                    if st != OK:
                        return st, []
                st, value, pos = self._literal(block, pos)
                if st != OK:
                    return st, []
            seen_field |= kind != SIZE_UPDATE
            records.append((kind, index) + field_strings(kind, index, name, value))
        return OK, records

    def decode_batch(self, data, offsets):
        """The arrays aws_hpack_header_block_decode_batch writes."""
        status, kinds, indices, strings = [], [], [], []
        field_offsets = [0]
        for i in range(len(offsets) - 1):
            st, recs = self.decode_block(bytes(data[int(offsets[i]):int(offsets[i + 1])]))
            status.append(st)
            for kind, index, name, value in recs:
                kinds.append(kind)
                indices.append(index)
                strings += [name, value]
            field_offsets.append(len(kinds))
        string_offsets = np.zeros(len(strings) + 1, dtype=np.uint64)
        string_offsets[1:] = np.cumsum([len(s) for s in strings])
        return {"field_offsets": np.array(field_offsets, dtype=np.uint64), "field_kind": np.array(kinds, dtype=np.uint8),
                "field_index": np.array(indices, dtype=np.uint64),
                "strings": np.frombuffer(b"".join(strings), dtype=np.uint8), "string_offsets": string_offsets,
                "status": np.array(status, dtype=np.int32)}

    # ---- encode ----
    def encode_field(self, name, value, never_indexed=False, mode=lit.SMALLEST):
        name, value = bytes(name), bytes(value)
        name_index = static_name_index(name)
        if never_indexed:
            head = lit.encode_integer(name_index, 4, 0x10)
        else:
            exact = static_exact_index(name, value)
            if exact:
                return lit.encode_integer(exact, 7, 0x80)
            head = lit.encode_integer(name_index, 4, 0x00)
        if not name_index:
            head += self.lit.encode(name, mode)
        return head + self.lit.encode(value, mode)

    def encode_batch(self, field_offsets, strings, string_offsets, never_indexed=None, mode=lit.SMALLEST):
        blocks = []
        for i in range(len(field_offsets) - 1):
            out = b""
            for f in range(int(field_offsets[i]), int(field_offsets[i + 1])):
                name = bytes(strings[int(string_offsets[2 * f]):int(string_offsets[2 * f + 1])])
                value = bytes(strings[int(string_offsets[2 * f + 1]):int(string_offsets[2 * f + 2])])
                out += self.encode_field(name, value, bool(never_indexed[f]) if never_indexed is not None else False, mode)
            blocks.append(out)
        offs = np.zeros(len(blocks) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(b) for b in blocks])
        return np.frombuffer(b"".join(blocks), dtype=np.uint8), offs

    # ---- random writer ----
    def random_block(self, rng, make_string, max_fields=12, long_values=(127, 255, 16511)):
        """A valid block with every representation kind, and the records a decoder returns for it.
        make_string(rng, length) -> bytes. Size updates (multi-byte ones too) only at the start; dynamic indices up
        to multi-byte values; empty names and values; a few values of `long_values` octets sent raw (so their
        length prefixes are 2, 3 and 4 octets long)."""
        out, records = b"", []
        for _ in range(int(rng.integers(0, 3)) if rng.random() < 0.3 else 0):
            size = int(rng.choice([0, 30, 4096, 1 << 20]))
            out += lit.encode_integer(size, 5, 0x20)
            records.append((SIZE_UPDATE, size, b"", b""))
        for _ in range(int(rng.integers(0, max_fields + 1))):
            kind = int(rng.choice([INDEXED, INCREMENTAL, WITHOUT, NEVER]))
            r = rng.random()
            if kind == INDEXED:
                index = int(rng.integers(1, 62)) if r < 0.6 else int(rng.choice([62, 63, 127, 128, 300, 70000]))
                out += lit.encode_integer(index, 7, 0x80)
                records.append((INDEXED, index) + field_strings(INDEXED, index))
                continue
            index = 0 if r < 0.4 else (int(rng.integers(1, 62)) if r < 0.8 else int(rng.choice([62, 63, 64, 100, 5000])))
            out += lit.encode_integer(index, _PREFIX[kind][0], _PREFIX[kind][1])
            name = b""
            if index == 0:
                name = make_string(rng, int(rng.integers(0, 24)))
                out += self.lit.encode(name, int(rng.integers(0, 3)))
            if rng.random() < 0.03:
                value = make_string(rng, int(rng.choice(long_values)))
                out += self.lit.encode(value, lit.NEVER)
            else:
                value = make_string(rng, int(rng.integers(0, 48)))
                out += self.lit.encode(value, int(rng.integers(0, 3)))
            records.append((kind, index) + field_strings(kind, index, name, value))
        return out, records
