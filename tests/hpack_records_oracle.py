"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

CPU restatement of the records encoder of aws_hpack_header_block_encode_records_batch, an encoder's side of the
HPACK dynamic table, and helpers, over the header-block oracle (oracle/hpack_header_block_oracle.py). Used only as the
checker by tests/test_hpack_header_block_records.py and as the record source of tools/header_blocks_probe.py.

Pinned on RFC 7541 Appendix C: the records the block oracle decodes from every C.2 to C.6 block encode back to the
RFC's octets, and the EncoderTable policy reproduces the RFC's own representations for C.3.1 to C.3.3, C.5.1, C.6.2
and C.6.3 (tests/test_hpack_header_block_records.py).

It holds:
  * RecordsOracle (a BlockOracle): encode_record / encode_records / encode_records_batch, the caller's kind and index
    per field, AUTO for the stateless rules, a status per block; random_block with an optional Huffman mode that
    frames every literal (None: the block oracle's writer as it is);
  * EncoderTable: an encoder-side dynamic table (RFC 7541 sections 2.3, 4) and the policy that turns a connection's
    header lists into records;
  * records_batch: record lists into the arrays of struct aws_hpack_header_lists.

Pure-Python loops; the table lookups are dictionaries, fast enough for the probe's millions of fields.
"""
import importlib.util
import os
from collections import deque

import numpy as np

_spec = importlib.util.spec_from_file_location(
    "hpack_header_block_oracle",
    os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "hpack_header_block_oracle.py"))
blk = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(blk)
lit = blk.lit

OK, INVALID_ARGUMENT = blk.OK, blk.INVALID_ARGUMENT
INDEXED, INCREMENTAL, WITHOUT, NEVER, SIZE_UPDATE = blk.INDEXED, blk.INCREMENTAL, blk.WITHOUT, blk.NEVER, blk.SIZE_UPDATE
AUTO = 5  # enum aws_hpack_field_kind: encode records only
_PREFIX, STATIC_TABLE, field_strings = blk._PREFIX, blk.STATIC_TABLE, blk.field_strings


class _FixedMode:
    """A literal oracle whose encode frames every literal in one Huffman mode, whatever mode it is asked for."""

    def __init__(self, literal_oracle, mode):
        self._lit, self._mode = literal_oracle, mode

    def encode(self, s, mode=None):
        return self._lit.encode(s, self._mode)

    def __getattr__(self, name):
        return getattr(self._lit, name)


class RecordsOracle(blk.BlockOracle):
    def encode_record(self, kind, index, name, value, never_indexed=False, mode=lit.SMALLEST):
        """The octets of one record, or None when the record is invalid on its own."""
        if kind == AUTO:
            return self.encode_field(name, value, never_indexed, mode)
        if kind not in _PREFIX or (kind == INDEXED and index == 0):
            return None
        bits, flags = _PREFIX[kind]
        if index - ((1 << bits) - 1) >= 1 << 63:  # more than 9 continuation octets: a decoder refuses it
            return None
        out = lit.encode_integer(index, bits, flags)
        if kind in (INCREMENTAL, WITHOUT, NEVER):
            if index == 0:
                out += self.lit.encode(bytes(name), mode)
            out += self.lit.encode(bytes(value), mode)
        return out

    def encode_records(self, records, never_indexed=None, mode=lit.SMALLEST):
        """(status, octets) of one block from records [(kind, index, name, value)]; an invalid block is empty."""
        out, seen_field = b"", False
        for f, (kind, index, name, value) in enumerate(records):
            if kind == SIZE_UPDATE and seen_field:
                return INVALID_ARGUMENT, b""
            seen_field |= kind != SIZE_UPDATE
            octets = self.encode_record(kind, index, name, value, bool(never_indexed[f]) if never_indexed is not None else False,
                                        mode)
            if octets is None:
                return INVALID_ARGUMENT, b""
            out += octets
        return OK, out

    def encode_records_batch(self, field_offsets, field_kind, field_index, strings, string_offsets, never_indexed=None,
                             mode=lit.SMALLEST):
        """(out, out_offsets, status) as aws_hpack_header_block_encode_records_batch writes them."""
        blocks, status = [], []
        for i in range(len(field_offsets) - 1):
            f0, f1 = int(field_offsets[i]), int(field_offsets[i + 1])
            records = [(int(field_kind[f]), int(field_index[f]),
                        bytes(strings[int(string_offsets[2 * f]):int(string_offsets[2 * f + 1])]),
                        bytes(strings[int(string_offsets[2 * f + 1]):int(string_offsets[2 * f + 2])]))
                       for f in range(f0, f1)]
            st, out = self.encode_records(records, None if never_indexed is None else never_indexed[f0:f1], mode)
            status.append(st)
            blocks.append(out)
        offs = np.zeros(len(blocks) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(b) for b in blocks])
        return np.frombuffer(b"".join(blocks), dtype=np.uint8), offs, np.array(status, dtype=np.int32)

    def random_block(self, rng, make_string, max_fields=12, long_values=(127, 255, 16511), mode=None):
        """The block oracle's random writer; with a mode, every literal is framed in it (the long values too). The
        random draws and the records are the same either way."""
        writer = self if mode is None else blk.BlockOracle(_FixedMode(self.lit, mode))
        return blk.BlockOracle.random_block(writer, rng, make_string, max_fields, long_values)


# ---- the encoder's side of the dynamic table ----
_STATIC_EXACT, _STATIC_NAME = {}, {}
for _i, (_n, _v) in enumerate(STATIC_TABLE):
    _STATIC_EXACT.setdefault((_n, _v), _i + 1)
    _STATIC_NAME.setdefault(_n, _i + 1)


class EncoderTable:
    """An encoder's dynamic table (RFC 7541 sections 2.3.2, 4: entry size = name + value + 32, the oldest entries
    evicted first) and the policy that picks each field's record, in this order:
        1. the (name, value) is in Appendix A                -> INDEXED, that index
        2. the (name, value) is in the dynamic table         -> INDEXED, 62 + its position (newest first)
        3. the name is in Appendix A                         -> LITERAL_INCREMENTAL with that name index
        4. the name is in the dynamic table                  -> LITERAL_INCREMENTAL with that name index
        5. otherwise                                         -> LITERAL_INCREMENTAL with a literal name
    Every INCREMENTAL field is inserted. A never-indexed field becomes LITERAL_NEVER_INDEXED (name index by rules 3,
    4, else 0) and is not inserted. A size change (set_max_size) becomes a TABLE_SIZE_UPDATE before the next list's
    first field (two when the size went down and back up: the lowest, then the last, RFC 7541 section 4.2).
    Records are in the decoder's form: (kind, index) + field_strings(...), so a decode of the encoded block returns
    them exactly. Lookups are dictionaries over insertion numbers, fast enough for a probe's millions of fields."""

    def __init__(self, max_size=4096):
        self.max_size, self.size = max_size, 0
        self.entries = deque()  # (insertion number, name, value), oldest on the left
        self.inserted = 0
        self.exact, self.names = {}, {}  # newest insertion number per (name, value) / name
        self.pending = None  # (lowest, last) size since the previous list

    def _evict(self, room):
        while self.entries and self.size > room:
            seq, name, value = self.entries.popleft()
            self.size -= 32 + len(name) + len(value)
            if self.exact.get((name, value)) == seq:  # the newest such entry is the last to go
                del self.exact[(name, value)]
            if self.names.get(name) == seq:
                del self.names[name]

    def _insert(self, name, value):
        size = 32 + len(name) + len(value)
        self._evict(self.max_size - size)
        if size > self.max_size:  # an entry larger than the table empties it and is not added
            return
        self.entries.append((self.inserted, name, value))
        self.exact[(name, value)] = self.names[name] = self.inserted
        self.inserted += 1
        self.size += size

    def _index(self, seq):
        return 62 + (self.inserted - 1 - seq)

    def set_max_size(self, max_size):
        low = max_size if self.pending is None else min(self.pending[0], max_size)
        self.pending = (low, max_size)
        self.max_size = max_size
        self._evict(max_size)

    def records(self, headers, never_indexed=()):
        """The records of one header list [(name, value)]; never_indexed: one flag per header (or empty)."""
        out = []
        if self.pending is not None:
            low, last = self.pending
            out += [(SIZE_UPDATE, low, b"", b"")] + ([(SIZE_UPDATE, last, b"", b"")] if last != low else [])
            self.pending = None
        for f, (name, value) in enumerate(headers):
            name, value = bytes(name), bytes(value)
            never = bool(never_indexed[f]) if len(never_indexed) else False
            index = 0 if never else _STATIC_EXACT.get((name, value), 0)
            if not index and not never and (name, value) in self.exact:
                index = self._index(self.exact[(name, value)])
            if index:
                out.append((INDEXED, index) + field_strings(INDEXED, index))
                continue
            name_index = _STATIC_NAME.get(name) or (self._index(self.names[name]) if name in self.names else 0)
            kind = NEVER if never else INCREMENTAL
            out.append((kind, name_index) + field_strings(kind, name_index, name, value))
            if kind == INCREMENTAL:
                self._insert(name, value)
        return out


def records_batch(blocks):
    """Record lists [(kind, index, name, value)] per block -> (field_offsets, field_kind, field_index, strings,
    string_offsets), the arrays of struct aws_hpack_header_lists."""
    records = [r for block in blocks for r in block]
    field_offsets = np.zeros(len(blocks) + 1, dtype=np.uint64)
    field_offsets[1:] = np.cumsum([len(b) for b in blocks])
    strings = [s for r in records for s in r[2:]]
    string_offsets = np.zeros(len(strings) + 1, dtype=np.uint64)
    string_offsets[1:] = np.cumsum([len(s) for s in strings])
    return (field_offsets, np.array([r[0] for r in records], dtype=np.uint8),
            np.array([r[1] for r in records], dtype=np.uint64), np.frombuffer(b"".join(strings), dtype=np.uint8),
            string_offsets)
