"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

CPU restatement of HPACK string literals (RFC 7541 sections 5.1 and 5.2) around the Huffman oracle
(oracle/huffman_oracle.c), used only as the checker by tests/ (SURVEY.md 8f.1).

Parity status: the reference repository (awslabs/aws-c-compression) holds NO framing code — the framing lives
in its caller, aws-c-http, which is absent from /root/reference. Pinned on the published algorithm instead:
RFC 7541 section 5.1 (prefix integers, Appendix C.1 worked examples), section 5.2 (string literals, padding rule)
and the string literals of Appendix C.2 / C.4 / C.6 (tests/test_hpack_literals.py::test_oracle_*). The Huffman
half is the pinned oracle. Against the reference itself: "parity unpinned" (nothing to pin to).

Pure-Python loops: fine for the test sizes (thousands of short strings).
"""
import numpy as np

OK = 0
SHORT_BUFFER = 4
INVALID_ARGUMENT = 34
UNKNOWN_SYMBOL = 3072
INVALID_PADDING = 3075

SMALLEST, NEVER, ALWAYS = 0, 1, 2


def encode_integer(value, prefix_bits, first_byte_flags=0):
    """RFC 7541 section 5.1."""
    limit = (1 << prefix_bits) - 1
    if value < limit:
        return bytes([first_byte_flags | value])
    out = [first_byte_flags | limit]
    value -= limit
    while value >= 128:
        out.append(value % 128 + 128)
        value //= 128
    out.append(value)
    return bytes(out)


def decode_integer(data, prefix_bits):
    """Returns (value, bytes used) or (None, status)."""
    if len(data) == 0:
        return None, SHORT_BUFFER
    limit = (1 << prefix_bits) - 1
    value = data[0] & limit
    used = 1
    if value < limit:
        return value, used
    shift = 0
    while True:
        if used >= len(data):
            return None, SHORT_BUFFER
        b = data[used]
        used += 1
        if shift > 56:
            return None, INVALID_ARGUMENT
        value += (b & 127) << shift
        shift += 7
        if not (b & 128):
            return value, used


class LiteralOracle:
    """huffman: a refcodec.OracleLib; table: its table for the code in use (RFC 7541 Appendix B for HPACK)."""

    def __init__(self, huffman, table, eos_padding=0xFF):
        self.h = huffman
        self.table = table
        self.eos = eos_padding

    def _huffman_encode(self, raw):
        raw = np.frombuffer(bytes(raw), dtype=np.uint8)
        offs = np.array([0, len(raw)], dtype=np.uint64)
        r = self.h.encode_batch(self.table, self.eos, raw, offs, out_capacity=4 * len(raw) + 8)
        return bytes(r["out"][:int(r["out_offsets"][1])])

    def encode(self, raw, mode=SMALLEST):
        raw = bytes(raw)
        if mode == NEVER:
            return encode_integer(len(raw), 7, 0x00) + raw
        enc = self._huffman_encode(raw)
        if mode == ALWAYS or len(enc) < len(raw):
            return encode_integer(len(enc), 7, 0x80) + enc
        return encode_integer(len(raw), 7, 0x00) + raw

    def decode(self, literal):
        """One literal exactly. Returns (status, string)."""
        literal = bytes(literal)
        length, used = decode_integer(literal, 7)
        if length is None:
            return used, b""
        huff = literal[0] >> 7
        rest = len(literal) - used
        if length > rest:
            return SHORT_BUFFER, b""
        if length < rest:
            return INVALID_ARGUMENT, b""
        payload = literal[used:]
        if not huff:
            return OK, payload
        dec = self.h.new_decoder(self.table)
        out = np.zeros(len(payload) * 8 + 8, dtype=np.uint8)  # (a code of 1 bit: eight symbols per octet)
        rc, _, olen = self.h.decode_call(dec, np.frombuffer(payload, dtype=np.uint8), out, 0, len(out))
        if rc != OK:
            return rc, b""
        # section 5.2: padding strictly shorter than a byte, the most significant bits of EOS (all ones); the
        # decoder's leftover register holds exactly the bits that matched no symbol (reference README.md:176-183)
        nb = dec.num_bits
        if nb >= 8:
            return INVALID_PADDING, b""
        if nb and (dec.working_bits >> (64 - nb)) != (1 << nb) - 1:
            return INVALID_PADDING, b""
        return OK, bytes(out[:olen])

    def encode_batch(self, data, offsets, mode=SMALLEST):
        outs = [self.encode(bytes(data[int(offsets[i]):int(offsets[i + 1])]), mode) for i in range(len(offsets) - 1)]
        offs = np.zeros(len(outs) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(o) for o in outs])
        return np.frombuffer(b"".join(outs), dtype=np.uint8), offs

    def decode_batch(self, data, offsets):
        status, outs = [], []
        for i in range(len(offsets) - 1):
            st, s = self.decode(bytes(data[int(offsets[i]):int(offsets[i + 1])]))
            status.append(st)
            outs.append(s if st == OK else b"")
        offs = np.zeros(len(outs) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(o) for o in outs])
        return np.frombuffer(b"".join(outs), dtype=np.uint8), offs, np.array(status, dtype=np.int32)
