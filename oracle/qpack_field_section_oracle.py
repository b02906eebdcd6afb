"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

CPU restatement of QPACK field sections (RFC 9204 section 4.5: the field section prefix and the five field line
formats, the Appendix A static table) over the literal oracle (oracle/hpack_literals_oracle.py: its prefix integers
and its Huffman code, which RFC 9204 4.1 takes from RFC 7541), used only as the checker by
tests/test_qpack_field_sections.py. The N-bit-prefix name literal (H at bit 3, 3-bit length) is framed here.

Parity status: unpinned against the reference — the reference repository (awslabs/aws-c-compression) holds no QPACK
code. Pinned on RFC 9204 instead: the field sections of Appendix B decode to the RFC's field lines and, through a
dynamic table kept by the test, to the RFC's header lists.

It holds:
  * STATIC_TABLE (Appendix A, 99 entries, 2026 octets of names and values);
  * SectionOracle.decode_section / decode_batch: the decode semantics of aws_qpack_field_section_decode_batch (the
    prefix as on the wire, one record per field line, static references resolved, dynamic and post-base references
    reported with empty strings, the first error a front-to-back decoder meets, nothing for a failing section);
  * SectionOracle.encode_field / encode_batch: the stateless encoder's rules;
  * SectionOracle.encode_records_batch: the records encoder, with its section rules;
  * SectionOracle.random_section: a writer that emits every line kind, with the records a decoder must return.

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
(INDEXED_STATIC, INDEXED_DYNAMIC, INDEXED_POST_BASE, NAME_REF_STATIC, NAME_REF_DYNAMIC, NAME_REF_POST_BASE,
 LITERAL_NAME, AUTO) = range(8)
# (prefix bits, first-octet flags, N flag) per line kind
_LINE = {INDEXED_STATIC: (6, 0xC0, 0), INDEXED_DYNAMIC: (6, 0x80, 0), INDEXED_POST_BASE: (4, 0x10, 0),
         NAME_REF_STATIC: (4, 0x50, 0x20), NAME_REF_DYNAMIC: (4, 0x40, 0x20), NAME_REF_POST_BASE: (3, 0x00, 0x08),
         LITERAL_NAME: (3, 0x20, 0x10)}
DYNAMIC_KINDS = {INDEXED_DYNAMIC, INDEXED_POST_BASE, NAME_REF_DYNAMIC, NAME_REF_POST_BASE}
STATIC_KINDS = {INDEXED_STATIC, NAME_REF_STATIC}
INDEXED_KINDS = {INDEXED_STATIC, INDEXED_DYNAMIC, INDEXED_POST_BASE}

STATIC_TABLE = [(n.encode(), v.encode()) for n, v in [
    (":authority", ""), (":path", "/"), ("age", "0"), ("content-disposition", ""), ("content-length", "0"),
    ("cookie", ""), ("date", ""), ("etag", ""), ("if-modified-since", ""), ("if-none-match", ""),
    ("last-modified", ""), ("link", ""), ("location", ""), ("referer", ""), ("set-cookie", ""),
    (":method", "CONNECT"), (":method", "DELETE"), (":method", "GET"), (":method", "HEAD"), (":method", "OPTIONS"),
    (":method", "POST"), (":method", "PUT"), (":scheme", "http"), (":scheme", "https"), (":status", "103"),
    (":status", "200"), (":status", "304"), (":status", "404"), (":status", "503"), ("accept", "*/*"),
    ("accept", "application/dns-message"), ("accept-encoding", "gzip, deflate, br"), ("accept-ranges", "bytes"),
    ("access-control-allow-headers", "cache-control"), ("access-control-allow-headers", "content-type"),
    ("access-control-allow-origin", "*"), ("cache-control", "max-age=0"), ("cache-control", "max-age=2592000"),
    ("cache-control", "max-age=604800"), ("cache-control", "no-cache"), ("cache-control", "no-store"),
    ("cache-control", "public, max-age=31536000"), ("content-encoding", "br"), ("content-encoding", "gzip"),
    ("content-type", "application/dns-message"), ("content-type", "application/javascript"),
    ("content-type", "application/json"), ("content-type", "application/x-www-form-urlencoded"),
    ("content-type", "image/gif"), ("content-type", "image/jpeg"), ("content-type", "image/png"),
    ("content-type", "text/css"), ("content-type", "text/html; charset=utf-8"), ("content-type", "text/plain"),
    ("content-type", "text/plain;charset=utf-8"), ("range", "bytes=0-"), ("strict-transport-security", "max-age=31536000"),
    ("strict-transport-security", "max-age=31536000; includesubdomains"),
    ("strict-transport-security", "max-age=31536000; includesubdomains; preload"), ("vary", "accept-encoding"),
    ("vary", "origin"), ("x-content-type-options", "nosniff"), ("x-xss-protection", "1; mode=block"),
    (":status", "100"), (":status", "204"), (":status", "206"), (":status", "302"), (":status", "400"),
    (":status", "403"), (":status", "421"), (":status", "425"), (":status", "500"), ("accept-language", ""),
    ("access-control-allow-credentials", "FALSE"), ("access-control-allow-credentials", "TRUE"),
    ("access-control-allow-headers", "*"), ("access-control-allow-methods", "get"),
    ("access-control-allow-methods", "get, post, options"), ("access-control-allow-methods", "options"),
    ("access-control-expose-headers", "content-length"), ("access-control-request-headers", "content-type"),
    ("access-control-request-method", "get"), ("access-control-request-method", "post"), ("alt-svc", "clear"),
    ("authorization", ""), ("content-security-policy", "script-src 'none'; object-src 'none'; base-uri 'none'"),
    ("early-data", "1"), ("expect-ct", ""), ("forwarded", ""), ("if-range", ""), ("origin", ""),
    ("purpose", "prefetch"), ("server", ""), ("timing-allow-origin", "*"), ("upgrade-insecure-requests", "1"),
    ("user-agent", ""), ("x-forwarded-for", ""), ("x-frame-options", "deny"), ("x-frame-options", "sameorigin")]]
assert len(STATIC_TABLE) == 99 and sum(len(n) + len(v) for n, v in STATIC_TABLE) == 2026


def static_name_index(name):
    """The lowest Appendix A index whose name is `name`, or None."""
    for i, (n, _) in enumerate(STATIC_TABLE):
        if n == name:
            return i
    return None


def static_exact_index(name, value):
    for i, entry in enumerate(STATIC_TABLE):
        if entry == (name, value):
            return i
    return None


def field_strings(kind, index, name=b"", value=b""):
    """The (name, value) a record carries: static references resolved, dynamic and post-base ones empty."""
    if kind == INDEXED_STATIC:
        return STATIC_TABLE[index]
    if kind in (INDEXED_DYNAMIC, INDEXED_POST_BASE):
        return b"", b""
    if kind == NAME_REF_STATIC:
        return STATIC_TABLE[index][0], value
    if kind in (NAME_REF_DYNAMIC, NAME_REF_POST_BASE):
        return b"", value
    return name, value


def int_refused(value, prefix_bits):
    """A decoder (hpack_read_int) refuses more than 9 continuation octets."""
    return len(lit.encode_integer(value, prefix_bits)) > 10


def encode_prefix(eic, sign, delta):
    return lit.encode_integer(eic, 8) + lit.encode_integer(delta, 7, 0x80 if sign else 0)


class SectionOracle:
    def __init__(self, literal_oracle):
        self.lit = literal_oracle

    # ---- literals ----
    def _literal(self, section, pos, prefix_bits, huff_mask):
        """(status, string, new pos) for the literal whose length integer starts at section[pos] (RFC 9204 4.1.2)."""
        if pos >= len(section):
            return SHORT_BUFFER, b"", pos
        length, used = lit.decode_integer(section[pos:], prefix_bits)
        if length is None:
            return used, b"", pos
        if length > len(section) - pos - used:
            return SHORT_BUFFER, b"", pos
        huff = section[pos] & huff_mask
        payload = section[pos + used:pos + used + length]
        # the literal oracle decodes RFC 7541 5.2 literals: the same payload behind H in bit 7 and a 7-bit length
        st, s = self.lit.decode(lit.encode_integer(length, 7, 0x80 if huff else 0) + payload)
        return st, s, pos + used + length

    def name_literal(self, name, mode, never):
        """001NH + 3-bit-prefix length + payload, the payload and H as `mode` frames the name."""
        framed = self.lit.encode(name, mode)
        length, used = lit.decode_integer(framed, 7)
        flags = 0x20 | (0x10 if never else 0) | (0x08 if framed[0] & 0x80 else 0)
        return lit.encode_integer(length, 3, flags) + framed[used:]

    # ---- decode ----
    def decode_section(self, section):
        """Returns (status, (eic, sign, delta), records) with records = [(kind, index, never, name, value)]; a zero
        prefix and no records when status != OK."""
        section = bytes(section)
        fail = lambda st: (st, (0, 0, 0), [])  # noqa: E731
        eic, used = lit.decode_integer(section, 8)
        if eic is None:
            return fail(used)
        pos = used
        if pos >= len(section):
            return fail(SHORT_BUFFER)
        sign = section[pos] >> 7
        delta, used = lit.decode_integer(section[pos:], 7)
        if delta is None:
            return fail(used)
        pos += used
        records = []
        while pos < len(section):
            b0 = section[pos]
            if b0 & 0x80:
                kind = INDEXED_STATIC if b0 & 0x40 else INDEXED_DYNAMIC
            elif b0 & 0x40:
                kind = NAME_REF_STATIC if b0 & 0x10 else NAME_REF_DYNAMIC
            elif b0 & 0x20:
                kind = LITERAL_NAME
            else:
                kind = INDEXED_POST_BASE if b0 & 0x10 else NAME_REF_POST_BASE
            bits, _, nflag = _LINE[kind]
            never = 1 if b0 & nflag else 0
            index, name, value = 0, b"", b""
            if kind == LITERAL_NAME:
                st, name, pos = self._literal(section, pos, 3, 0x08)
                if st != OK:
                    return fail(st)
            else:
                if eic == 0 and kind in DYNAMIC_KINDS:
                    return fail(INVALID_ARGUMENT)
                index, used = lit.decode_integer(section[pos:], bits)
                if index is None:
                    return fail(used)
                pos += used
                if kind in STATIC_KINDS and index >= len(STATIC_TABLE):
                    return fail(INVALID_ARGUMENT)
            if kind not in INDEXED_KINDS:
                st, value, pos = self._literal(section, pos, 7, 0x80)
                if st != OK:
                    return fail(st)
            records.append((kind, index, never) + field_strings(kind, index, name, value))
        return OK, (eic, sign, delta), records

    def decode_batch(self, data, offsets):
        """The arrays aws_qpack_field_section_decode_batch writes."""
        status, prefix, kinds, indices, nevers, strings = [], [], [], [], [], []
        field_offsets = [0]
        for i in range(len(offsets) - 1):
            st, pre, recs = self.decode_section(bytes(data[int(offsets[i]):int(offsets[i + 1])]))
            status.append(st)
            prefix.append(pre)
            for kind, index, never, name, value in recs:
                kinds.append(kind)
                indices.append(index)
                nevers.append(never)
                strings += [name, value]
            field_offsets.append(len(kinds))
        string_offsets = np.zeros(len(strings) + 1, dtype=np.uint64)
        string_offsets[1:] = np.cumsum([len(s) for s in strings])
        prefix = np.array(prefix, dtype=np.uint64).reshape(-1, 3)
        return {"encoded_insert_count": prefix[:, 0].copy(), "base_sign": prefix[:, 1].astype(np.uint8),
                "delta_base": prefix[:, 2].copy(), "field_offsets": np.array(field_offsets, dtype=np.uint64),
                "field_kind": np.array(kinds, dtype=np.uint8), "field_index": np.array(indices, dtype=np.uint64),
                "never_indexed": np.array(nevers, dtype=np.uint8),
                "strings": np.frombuffer(b"".join(strings), dtype=np.uint8), "string_offsets": string_offsets,
                "status": np.array(status, dtype=np.int32)}

    # ---- encode ----
    def encode_line(self, kind, index, never, name, value, mode=lit.SMALLEST):
        """One field line as the record says (kind not AUTO); None when the records encoder refuses it."""
        if kind > AUTO or (kind in STATIC_KINDS and index >= len(STATIC_TABLE)):
            return None
        if kind == LITERAL_NAME:
            length, _ = lit.decode_integer(self.lit.encode(name, mode), 7)
            if int_refused(length, 3):
                return None
            return self.name_literal(name, mode, never) + self.lit.encode(value, mode)
        bits, flags, nflag = _LINE[kind]
        if int_refused(index, bits):
            return None
        out = lit.encode_integer(index, bits, flags | (nflag if never else 0))
        return out if kind in INDEXED_KINDS else out + self.lit.encode(value, mode)

    def encode_field(self, name, value, never_indexed=False, mode=lit.SMALLEST):
        """The stateless rules."""
        name, value = bytes(name), bytes(value)
        name_index = static_name_index(name)
        if not never_indexed:
            exact = static_exact_index(name, value)
            if exact is not None:
                return self.encode_line(INDEXED_STATIC, exact, 0, name, value, mode)
        if name_index is not None:
            return self.encode_line(NAME_REF_STATIC, name_index, never_indexed, name, value, mode)
        return self.encode_line(LITERAL_NAME, 0, never_indexed, name, value, mode)

    @staticmethod
    def _fields(strings, string_offsets, f):
        return (bytes(strings[int(string_offsets[2 * f]):int(string_offsets[2 * f + 1])]),
                bytes(strings[int(string_offsets[2 * f + 1]):int(string_offsets[2 * f + 2])]))

    def encode_batch(self, field_offsets, strings, string_offsets, never_indexed=None, mode=lit.SMALLEST):
        sections = []
        for i in range(len(field_offsets) - 1):
            out = encode_prefix(0, 0, 0)
            for f in range(int(field_offsets[i]), int(field_offsets[i + 1])):
                name, value = self._fields(strings, string_offsets, f)
                out += self.encode_field(name, value, bool(never_indexed[f]) if never_indexed is not None else False, mode)
            sections.append(out)
        return _packed(sections)

    def encode_records_batch(self, eic, sign, delta, field_offsets, kinds, indices, strings, string_offsets,
                             never_indexed=None, mode=lit.SMALLEST):
        """(data, offsets, status) of aws_qpack_field_section_encode_records_batch."""
        sections, status = [], []
        for i in range(len(field_offsets) - 1):
            e, s, d = int(eic[i]), int(sign[i]), int(delta[i])
            ok = s in (0, 1) and not int_refused(e, 8) and not int_refused(d, 7)
            out = encode_prefix(e, s, d) if ok else b""
            for f in range(int(field_offsets[i]), int(field_offsets[i + 1])):
                if not ok:
                    break
                name, value = self._fields(strings, string_offsets, f)
                never = bool(never_indexed[f]) if never_indexed is not None else False
                kind = int(kinds[f])
                if kind == AUTO:
                    line = self.encode_field(name, value, never, mode)
                elif e == 0 and kind in DYNAMIC_KINDS:
                    line = None
                else:
                    line = self.encode_line(kind, int(indices[f]), never, name, value, mode)
                ok = line is not None
                out += line or b""
            sections.append(out if ok else b"")
            status.append(OK if ok else INVALID_ARGUMENT)
        data, offs = _packed(sections)
        return data, offs, np.array(status, dtype=np.int32)

    # ---- random writer ----
    def random_section(self, rng, make_string, max_fields=12, mode=None):
        """A valid section with every line kind, its prefix and the records a decoder returns for it.
        make_string(rng, length) -> bytes. Multi-octet integers at every prefix width (the 8- and 7-bit prefix
        integers, 6-, 4- and 3-bit indices, 3-bit name lengths of 7 and more), literal lengths of 1, 2 and 3 octets,
        N set and clear, Huffman and raw literals (mode None: a random mode per literal, else `mode` for all)."""
        pick = lambda: int(rng.integers(0, 3)) if mode is None else mode  # noqa: E731
        eic = 0 if rng.random() < 0.25 else int(rng.choice([1, 5, 200, 254, 255, 300, 70000]))
        sign = int(rng.integers(0, 2))
        delta = int(rng.choice([0, 1, 3, 126, 127, 500, 20000]))
        out, records = encode_prefix(eic, sign, delta), []
        kinds = [INDEXED_STATIC, NAME_REF_STATIC, LITERAL_NAME] + (sorted(DYNAMIC_KINDS) if eic else [])
        for _ in range(int(rng.integers(0, max_fields + 1))):
            kind = int(rng.choice(kinds))
            never = int(rng.random() < 0.3) if kind not in INDEXED_KINDS else 0
            if kind in STATIC_KINDS:
                index = int(rng.integers(0, 99))
            else:
                index = int(rng.integers(0, 20)) if rng.random() < 0.7 else int(rng.choice([62, 63, 127, 300, 70000]))
            name, value = b"", b""
            if kind == LITERAL_NAME:
                index = 0
                name = make_string(rng, int(rng.choice([0, 3, 6, 7, 20, 134, 135, 300])) if rng.random() < 0.3
                                   else int(rng.integers(0, 24)))
            if kind not in INDEXED_KINDS:
                value = make_string(rng, int(rng.choice([126, 127, 254, 255, 16511])) if rng.random() < 0.03
                                    else int(rng.integers(0, 48)))
            line = lit.encode_integer(index, _LINE[kind][0], _LINE[kind][1] | (_LINE[kind][2] if never else 0)) \
                if kind != LITERAL_NAME else self.name_literal(name, pick(), never)
            if kind not in INDEXED_KINDS:
                line += self.lit.encode(value, pick())
            out += line
            records.append((kind, index, never) + field_strings(kind, index, name, value))
        return out, (eic, sign, delta), records


def _packed(items):
    offs = np.zeros(len(items) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(b) for b in items])
    return np.frombuffer(b"".join(items), dtype=np.uint8), offs
