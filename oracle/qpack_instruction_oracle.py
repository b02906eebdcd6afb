"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

CPU restatement of QPACK's encoder- and decoder-stream instructions (RFC 9204 sections 4.3 and 4.4) over the literal
oracle (oracle/hpack_literals_oracle.py: prefix integers and the Huffman code) and the static table of
oracle/qpack_field_section_oracle.py, used only as the checker by tests/test_qpack_instructions.py. The
5-bit-prefix name literal (H at 0x20) is framed here.

Parity status: unpinned against the reference — the reference repository (awslabs/aws-c-compression) holds no QPACK
code. Pinned on RFC 9204 instead: the encoder- and decoder-stream octets of Appendix B decode to the RFC's
instructions, and those inserts, applied to a table kept by the test, resolve the appendix's field sections.

It holds:
  * InstructionOracle.decode_chunk / decode_batch: the decode semantics of aws_qpack_instruction_decode_batch (one
    record per instruction read in full, a chunk that ends inside an instruction is cut there and reports its consumed
    octets, the first error a front-to-back decoder meets, nothing for a failing chunk);
  * InstructionOracle.encode_instruction / encode_batch: the encoder, with its chunk rules;
  * InstructionOracle.random_stream: a writer that emits every instruction kind of a stream, with its records.

Pure-Python loops: fine for the test sizes.
"""
import importlib.util
import os

import numpy as np

_spec = importlib.util.spec_from_file_location(
    "qpack_field_section_oracle",
    os.path.join(os.path.dirname(os.path.abspath(__file__)), "qpack_field_section_oracle.py"))
sections = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(sections)
lit = sections.lit

OK, SHORT_BUFFER, INVALID_ARGUMENT = lit.OK, lit.SHORT_BUFFER, lit.INVALID_ARGUMENT
STATIC_TABLE = sections.STATIC_TABLE
ENCODER_STREAM, DECODER_STREAM = 0, 1
(INSERT_NAME_REF_STATIC, INSERT_NAME_REF_DYNAMIC, INSERT_LITERAL_NAME, DUPLICATE, SET_CAPACITY,
 SECTION_ACKNOWLEDGMENT, STREAM_CANCELLATION, INSERT_COUNT_INCREMENT, INSERT_AUTO) = range(9)
# (prefix bits, first-octet flags) per kind
FORMAT = {INSERT_NAME_REF_STATIC: (6, 0xC0), INSERT_NAME_REF_DYNAMIC: (6, 0x80), INSERT_LITERAL_NAME: (5, 0x40),
          DUPLICATE: (5, 0x00), SET_CAPACITY: (5, 0x20), SECTION_ACKNOWLEDGMENT: (7, 0x80),
          STREAM_CANCELLATION: (6, 0x40), INSERT_COUNT_INCREMENT: (6, 0x00)}
STREAM_KINDS = {ENCODER_STREAM: (INSERT_NAME_REF_STATIC, INSERT_NAME_REF_DYNAMIC, INSERT_LITERAL_NAME, DUPLICATE,
                                 SET_CAPACITY),
                DECODER_STREAM: (SECTION_ACKNOWLEDGMENT, STREAM_CANCELLATION, INSERT_COUNT_INCREMENT)}
INSERT_KINDS = (INSERT_NAME_REF_STATIC, INSERT_NAME_REF_DYNAMIC, INSERT_LITERAL_NAME)


def instruction_kind(which, b0):
    if which == ENCODER_STREAM:
        if b0 & 0x80:
            return INSERT_NAME_REF_STATIC if b0 & 0x40 else INSERT_NAME_REF_DYNAMIC
        if b0 & 0x40:
            return INSERT_LITERAL_NAME
        return SET_CAPACITY if b0 & 0x20 else DUPLICATE
    if b0 & 0x80:
        return SECTION_ACKNOWLEDGMENT
    return STREAM_CANCELLATION if b0 & 0x40 else INSERT_COUNT_INCREMENT


def instruction_strings(kind, index, name=b"", value=b""):
    """The (name, value) a record carries: the static name resolved, the dynamic one empty."""
    if kind == INSERT_NAME_REF_STATIC:
        return STATIC_TABLE[index][0], value
    if kind == INSERT_NAME_REF_DYNAMIC:
        return b"", value
    if kind == INSERT_LITERAL_NAME:
        return name, value
    return b"", b""


def _span(chunk, pos, prefix_bits, huff_mask):
    """(status, (H, payload), new pos) of the literal whose length integer starts at chunk[pos]; structure only."""
    if pos >= len(chunk):
        return SHORT_BUFFER, None, pos
    length, used = lit.decode_integer(chunk[pos:], prefix_bits)
    if length is None:
        return used, None, pos
    if length > len(chunk) - pos - used:
        return SHORT_BUFFER, None, pos
    return OK, (chunk[pos] & huff_mask, chunk[pos + used:pos + used + length]), pos + used + length


class InstructionOracle:
    def __init__(self, literal_oracle):
        self.lit = literal_oracle

    def _decode_span(self, span):
        huff, payload = span
        return self.lit.decode(lit.encode_integer(len(payload), 7, 0x80 if huff else 0) + payload)

    # ---- decode ----
    def decode_chunk(self, which, chunk):
        """Returns (status, consumed, records) with records = [(kind, index, name, value)]; consumed 0 and no
        records when status != OK."""
        chunk = bytes(chunk)
        fail = lambda st: (st, 0, [])  # noqa: E731
        pos, records = 0, []
        while pos < len(chunk):
            start = pos
            kind = instruction_kind(which, chunk[pos])
            index, name_span, value_span = 0, None, None
            if kind == INSERT_LITERAL_NAME:
                st, name_span, pos = _span(chunk, pos, 5, 0x20)
            else:
                index, used = lit.decode_integer(chunk[pos:], FORMAT[kind][0])
                st = OK if index is not None else used
                if index is not None:
                    pos += used
                    if (kind == INSERT_NAME_REF_STATIC and index >= len(STATIC_TABLE)) or \
                            (kind == INSERT_COUNT_INCREMENT and index == 0):
                        st = INVALID_ARGUMENT
            if st == OK and kind in INSERT_KINDS:
                st, value_span, pos = _span(chunk, pos, 7, 0x80)
            if st == SHORT_BUFFER:  # cut: nothing of this instruction, its name literal included
                return OK, start, records
            name, value = b"", b""
            if name_span is not None:  # (read in full: decoded, and its errors come first)
                name_st, name = self._decode_span(name_span)
                if name_st != OK:
                    return fail(name_st)
            if st != OK:
                return fail(st)
            if value_span is not None:
                value_st, value = self._decode_span(value_span)
                if value_st != OK:
                    return fail(value_st)
            records.append((kind, index) + instruction_strings(kind, index, name, value))
        return OK, pos, records

    def decode_batch(self, which, data, offsets):
        """The arrays aws_qpack_instruction_decode_batch writes."""
        status, consumed, kinds, indices, strings = [], [], [], [], []
        instruction_offsets = [0]
        for i in range(len(offsets) - 1):
            st, used, recs = self.decode_chunk(which, bytes(data[int(offsets[i]):int(offsets[i + 1])]))
            status.append(st)
            consumed.append(used)
            for kind, index, name, value in recs:
                kinds.append(kind)
                indices.append(index)
                strings += [name, value]
            instruction_offsets.append(len(kinds))
        string_offsets = np.zeros(len(strings) + 1, dtype=np.uint64)
        string_offsets[1:] = np.cumsum([len(s) for s in strings])
        return {"instruction_offsets": np.array(instruction_offsets, dtype=np.uint64),
                "kind": np.array(kinds, dtype=np.uint8), "index": np.array(indices, dtype=np.uint64),
                "strings": np.frombuffer(b"".join(strings), dtype=np.uint8), "string_offsets": string_offsets,
                "consumed": np.array(consumed, dtype=np.uint64), "status": np.array(status, dtype=np.int32)}

    # ---- encode ----
    def name_literal(self, name, mode):
        """01H + 5-bit-prefix length + payload, the payload and H as `mode` frames the name; None when the length is
        an integer a decoder refuses."""
        framed = self.lit.encode(name, mode)
        length, used = lit.decode_integer(framed, 7)
        if sections.int_refused(length, 5):
            return None
        return lit.encode_integer(length, 5, 0x40 | (0x20 if framed[0] & 0x80 else 0)) + framed[used:]

    def encode_instruction(self, which, kind, index, name=b"", value=b"", mode=lit.SMALLEST):
        """One instruction as the record says; None when the encoder refuses it."""
        name, value = bytes(name), bytes(value)
        if kind == INSERT_AUTO and which == ENCODER_STREAM:
            match = sections.static_name_index(name)
            kind, index = (INSERT_NAME_REF_STATIC, match) if match is not None else (INSERT_LITERAL_NAME, 0)
        if kind not in STREAM_KINDS[which]:
            return None
        if (kind == INSERT_NAME_REF_STATIC and index >= len(STATIC_TABLE)) or \
                (kind == INSERT_COUNT_INCREMENT and index == 0):
            return None
        if kind == INSERT_LITERAL_NAME:
            out = self.name_literal(name, mode)
        else:
            bits, flags = FORMAT[kind]
            out = None if sections.int_refused(index, bits) else lit.encode_integer(index, bits, flags)
        if out is None:
            return None
        return out + self.lit.encode(value, mode) if kind in INSERT_KINDS else out

    def encode_batch(self, which, instruction_offsets, kinds, indices, strings, string_offsets, mode=lit.SMALLEST):
        """(data, offsets, status) of aws_qpack_instruction_encode_batch."""
        chunks, status = [], []
        for i in range(len(instruction_offsets) - 1):
            out = b""
            for f in range(int(instruction_offsets[i]), int(instruction_offsets[i + 1])):
                name, value = b"", b""
                if which == ENCODER_STREAM:
                    name = bytes(strings[int(string_offsets[2 * f]):int(string_offsets[2 * f + 1])])
                    value = bytes(strings[int(string_offsets[2 * f + 1]):int(string_offsets[2 * f + 2])])
                line = self.encode_instruction(which, int(kinds[f]), int(indices[f]), name, value, mode)
                if line is None:
                    out = None
                    break
                out += line
            chunks.append(out or b"")
            status.append(OK if out is not None else INVALID_ARGUMENT)
        offs = np.zeros(len(chunks) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(c) for c in chunks])
        return np.frombuffer(b"".join(chunks), dtype=np.uint8), offs, np.array(status, dtype=np.int32)

    # ---- random writer ----
    def random_stream(self, rng, which, make_string, count, mode=None):
        """(octets, records) of `count` valid instructions of one stream, every kind of it: multi-octet integers at
        every prefix width (indices, capacities, stream IDs, 5-bit name lengths of 31 and more), literal lengths of 1,
        2 and 3 octets, Huffman and raw literals (mode None: a random mode per literal, else `mode` for all).
        make_string(rng, length) -> bytes."""
        pick = lambda: int(rng.integers(0, 3)) if mode is None else mode  # noqa: E731
        kinds = STREAM_KINDS[which]
        out, records = b"", []
        for _ in range(count):
            kind = int(rng.choice(kinds))
            if kind == INSERT_NAME_REF_STATIC:
                index = int(rng.integers(0, 99))
            elif kind == INSERT_LITERAL_NAME:
                index = 0
            else:
                index = int(rng.integers(0, 40)) if rng.random() < 0.7 else int(rng.choice([62, 63, 127, 300, 70000]))
                if kind == INSERT_COUNT_INCREMENT:
                    index = max(index, 1)
            name = make_string(rng, int(rng.choice([0, 3, 30, 31, 40, 300])) if rng.random() < 0.3
                               else int(rng.integers(0, 24))) if kind == INSERT_LITERAL_NAME else b""
            value = b""
            if kind in INSERT_KINDS:
                value = make_string(rng, int(rng.choice([126, 127, 254, 255, 16511])) if rng.random() < 0.03
                                    else int(rng.integers(0, 48)))
            line = self.name_literal(name, pick()) if kind == INSERT_LITERAL_NAME else \
                lit.encode_integer(index, *FORMAT[kind])
            if kind in INSERT_KINDS:
                line += self.lit.encode(value, pick())
            out += line
            records.append((kind, index) + instruction_strings(kind, index, name, value))
        return out, records
