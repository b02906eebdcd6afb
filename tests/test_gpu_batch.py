"""GPU parity: aws_huffman_encode_batch / aws_huffman_decode_batch (through the C ABI) against the
oracle on the same seeded inputs, bit for bit — bytes, lengths, offsets, status, cursor positions and
leftover encoder/decoder state — plus the committed outputs of the unmodified reference."""
import numpy as np
import pytest

import refcodec
from refcodec import OK, SHORT_BUFFER, UNKNOWN_SYMBOL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def contexts(pkg, coders):
    made = {}

    def get(table, eos=0xFF):
        key = (table, eos)
        if key not in made:
            made[key] = pkg.BatchContext(coders.coder(table), eos_padding=eos, device=0)
        return made[key]

    yield get
    for ctx in made.values():
        ctx.close()


def assert_same(got, want, keys=None, total_key="out_offsets"):
    for k in (keys or want.keys()):
        if k == "out":
            continue
        assert np.array_equal(got[k], want[k]), "%s differs (first at %s)" % (
            k, np.flatnonzero(np.asarray(got[k]) != np.asarray(want[k]))[:5])


def assert_same_packed(got, want):
    assert_same(got, want)
    total = int(want["out_offsets"][-1])
    assert np.array_equal(got["out"][:total], want["out"][:total]), "payload bytes differ"


def assert_same_slotted(got, want, slots):
    assert_same(got, want)
    for i in np.random.default_rng(1).permutation(len(slots))[:4000]:
        a, l = int(slots[i]), int(want["out_lens"][i])
        assert np.array_equal(got["out"][a:a + l], want["out"][a:a + l]), "item %d bytes differ" % i


def test_reference_golden_vectors_through_the_batch_api(contexts):
    g = refcodec.golden("reference_vectors.json")
    ctx = contexts("test")
    ins = [bytes.fromhex(k["input_hex"]) for k in g["encode_kats"]] + [b"cdfh", b""]
    want = [bytes.fromhex(k["encoded_hex"]) for k in g["encode_kats"]] + [bytes.fromhex("8218a3"), b""]
    data = np.frombuffer(b"".join(ins), dtype=np.uint8)
    offs = np.cumsum([0] + [len(x) for x in ins]).astype(np.uint64)
    enc = ctx.encode(data, offs, 1024)
    assert np.array_equal(enc["out_lens"], [len(w) for w in want])
    assert bytes(enc["out"][:int(enc["out_offsets"][-1])]) == b"".join(want)
    assert np.array_equal(ctx.encoded_lengths(data, offs), [len(w) for w in want])
    dec = ctx.decode(enc["out"][:int(enc["out_offsets"][-1])], enc["out_offsets"], 1024)
    assert np.array_equal(dec["out_offsets"], offs)
    assert bytes(dec["out"][:len(data)]) == b"".join(ins)
    assert (dec["status"] == OK).all() and (enc["status"] == OK).all()


def test_rfc7541_vectors(contexts):
    from test_oracle_pins import RFC7541_C
    ctx = contexts("hpack")
    data = np.frombuffer(b"".join(t for t, _ in RFC7541_C), dtype=np.uint8)
    offs = np.cumsum([0] + [len(t) for t, _ in RFC7541_C]).astype(np.uint64)
    enc = ctx.encode(data, offs, 4096)
    assert bytes(enc["out"][:int(enc["out_offsets"][-1])]).hex() == "".join(h for _, h in RFC7541_C)


@pytest.mark.parametrize("table_name", ["test", "hpack"])
def test_committed_reference_outputs(contexts, pkg, table_name):
    """Same fixture as the oracle pin test, now through the GPU: outputs of the unmodified reference."""
    cases = refcodec.golden("differential_%s.json" % table_name)
    plain = [c for c in cases["encode"] if not c["masked"]]
    by_eos = {}
    for c in plain:
        by_eos.setdefault(c["eos"], []).append(c)
    for eos, group in by_eos.items():
        ctx = contexts(table_name, eos)
        ins = [bytes.fromhex(c["in"]) for c in group]
        data = np.frombuffer(b"".join(ins), dtype=np.uint8)
        offs = np.cumsum([0] + [len(x) for x in ins]).astype(np.uint64)
        caps = np.array([c["cap"] for c in group], dtype=np.uint64)
        slots = np.zeros(len(group), dtype=np.uint64)
        slots[1:] = np.cumsum(caps)[:-1]
        r = ctx.encode(data, offs, int(caps.sum()) + 1, out_offsets=slots, out_caps=caps)
        for i, c in enumerate(group):
            a, l = int(slots[i]), int(r["out_lens"][i])
            assert bytes(r["out"][a:a + l]).hex() == c["out"]
            assert (int(r["status"][i]), int(r["consumed"][i]), int(r["overflow_pattern"][i]),
                    int(r["overflow_num_bits"][i])) == (c["status"], c["consumed"], c["ovf_pattern"], c["ovf_bits"])
    ctx = contexts(table_name)
    group = cases["decode"]
    ins = [bytes.fromhex(c["in"]) for c in group]
    data = np.frombuffer(b"".join(ins), dtype=np.uint8)
    offs = np.cumsum([0] + [len(x) for x in ins]).astype(np.uint64)
    caps = np.array([c["cap"] for c in group], dtype=np.uint64)
    slots = np.zeros(len(group), dtype=np.uint64)
    slots[1:] = np.cumsum(caps)[:-1]
    r = ctx.decode(data, offs, int(caps.sum()) + 1, out_offsets=slots, out_caps=caps)
    for i, c in enumerate(group):
        a, l = int(slots[i]), int(r["out_lens"][i])
        assert bytes(r["out"][a:a + l]).hex() == c["out"]
        assert (int(r["status"][i]), int(r["consumed"][i]), int(r["leftover_working_bits"][i]),
                int(r["leftover_num_bits"][i])) == (c["status"], c["consumed"], c["left_bits"], c["left_num"])


@pytest.mark.parametrize("table_name", ["test", "hpack"])
@pytest.mark.parametrize("zipf", [True, False])
def test_random_batches_match_oracle(contexts, oracle, oracle_tables, table_name, zipf):
    rng = np.random.default_rng(0xB200 + zipf)
    ctx, table = contexts(table_name), oracle_tables[table_name]
    data, offs = refcodec.random_batch(rng, 20000, 0, 300, table_name, zipf=zipf)
    n = len(offs) - 1
    cap_total = 4 * len(data) + 16
    want = oracle.encode_batch(table, 0xFF, data, offs, cap_total)
    got = ctx.encode(data, offs, cap_total)
    assert_same_packed(got, want)
    assert np.array_equal(ctx.encoded_lengths(data, offs), want["out_lens"])

    # slotted: capacities scattered around what each item needs
    caps = np.maximum(0, want["out_lens"].astype(np.int64) + rng.integers(-8, 3, size=n)).astype(np.uint64)
    slots = np.zeros(n, dtype=np.uint64)
    slots[1:] = np.cumsum(caps)[:-1]
    total = int(caps.sum()) + 1
    sentinel = np.full(total, 0xA5, dtype=np.uint8)
    want_s = oracle.encode_batch(table, 0xFF, data, offs, total, out_offsets=slots, out_caps=caps, out=sentinel.copy())
    got_s = ctx.encode(data, offs, total, out_offsets=slots, out_caps=caps, out=sentinel.copy())
    assert_same_slotted(got_s, want_s, slots)
    assert np.array_equal(got_s["out"], want_s["out"]), "bytes outside the written prefixes must stay untouched"
    assert (want_s["status"] == SHORT_BUFFER).any() and (want_s["status"] == OK).any()

    # decode what was encoded (packed), then with limited capacities
    stream = want["out"][:int(want["out_offsets"][-1])]
    want_d = oracle.decode_batch(table, stream, want["out_offsets"], len(data) + 16)
    got_d = ctx.decode(stream, want["out_offsets"], len(data) + 16)
    assert_same_packed(got_d, want_d)
    assert np.array_equal(got_d["out"][:len(data)], data)
    caps = np.maximum(0, want_d["out_lens"].astype(np.int64) + rng.integers(-6, 2, size=n)).astype(np.uint64)
    slots = np.zeros(n, dtype=np.uint64)
    slots[1:] = np.cumsum(caps)[:-1]
    total = int(caps.sum()) + 1
    want_ds = oracle.decode_batch(table, stream, want["out_offsets"], total, out_offsets=slots, out_caps=caps)
    got_ds = ctx.decode(stream, want["out_offsets"], total, out_offsets=slots, out_caps=caps)
    assert_same_slotted(got_ds, want_ds, slots)


@pytest.mark.parametrize("table_name", ["test", "hpack"])
def test_decode_of_arbitrary_bytes_matches_oracle(contexts, oracle, oracle_tables, table_name):
    """The reference's decode fuzzer (tests/fuzz/decode.c) as a differential test."""
    rng = np.random.default_rng(0xF022)
    ctx, table = contexts(table_name), oracle_tables[table_name]
    lens = rng.integers(0, 120, size=20000)
    offs = np.zeros(len(lens) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(lens)
    payload = rng.integers(0, 256, size=int(offs[-1]), dtype=np.uint8)
    payload[rng.random(len(payload)) < 0.3] = 0xFF  # long runs of ones reach the deep / invalid codes
    cap = 2 * len(payload) + 16
    want = oracle.decode_batch(table, payload, offs, cap)
    got = ctx.decode(payload, offs, cap)
    assert_same_packed(got, want)
    assert (want["status"] == UNKNOWN_SYMBOL).any() and (want["status"] == OK).any()


def test_unknown_symbols_on_encode(pkg, oracle, ref_free_masked_coder):
    """A coder whose ENCODE table has holes: UNKNOWN_SYMBOL, truncated lengths, cursor past the symbol."""
    coder, patterns, num_bits = ref_free_masked_coder
    ctx = pkg.BatchContext(coder, device=0)
    table = oracle.table(patterns, num_bits)
    rng = np.random.default_rng(5)
    data, offs = refcodec.random_batch(rng, 8000, 0, 120, "test", zipf=False)
    cap_total = 4 * len(data) + 16
    want = oracle.encode_batch(table, 0x3C, data, offs, cap_total)
    ctx2 = pkg.BatchContext(coder, eos_padding=0x3C, device=0)
    got = ctx2.encode(data, offs, cap_total)
    assert_same_packed(got, want)
    assert (want["status"] == UNKNOWN_SYMBOL).sum() > 100
    n = len(offs) - 1
    caps = np.maximum(0, want["out_lens"].astype(np.int64) + rng.integers(-4, 3, size=n)).astype(np.uint64)
    slots = np.zeros(n, dtype=np.uint64)
    slots[1:] = np.cumsum(caps)[:-1]
    total = int(caps.sum()) + 1
    want_s = oracle.encode_batch(table, 0x3C, data, offs, total, out_offsets=slots, out_caps=caps)
    got_s = ctx2.encode(data, offs, total, out_offsets=slots, out_caps=caps)
    assert_same_slotted(got_s, want_s, slots)
    ctx.close()
    ctx2.close()


def test_full_range_code_lengths(pkg, oracle):
    """Codes of 1, 31 and 32 bits (reference MAX_PATTERN_BITS, huffman.c:10; SURVEY.md App. B.1)."""
    import ctypes as C
    capi = pkg.capi
    patterns = np.zeros(256, dtype=np.uint32)
    num_bits = np.zeros(256, dtype=np.uint8)
    # 0 -> '0' (1 bit); 1 -> '10'; 2 -> 110 + 28 zeros (31 bits); 3 -> 111 + 29 zeros (32); 4 -> 111 + 28 zeros + 1 (32)
    patterns[0], num_bits[0] = 0b0, 1
    patterns[1], num_bits[1] = 0b10, 2
    patterns[2], num_bits[2] = 0b110 << 28, 31
    patterns[3], num_bits[3] = 0b111 << 29, 32
    patterns[4], num_bits[4] = (0b111 << 29) | 1, 32
    table = oracle.table(patterns, num_bits)

    coder = capi.python_coder(lambda sym: (patterns[sym], num_bits[sym]))
    ctx = pkg.BatchContext(coder, eos_padding=0xFF, device=0)
    rng = np.random.default_rng(11)
    lens = rng.integers(0, 200, size=3000)
    offs = np.zeros(len(lens) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(lens)
    data = rng.integers(0, 5, size=int(offs[-1])).astype(np.uint8)
    cap_total = 4 * len(data) + 16
    want = oracle.encode_batch(table, 0xFF, data, offs, cap_total)
    got = ctx.encode(data, offs, cap_total)
    assert_same_packed(got, want)
    stream = want["out"][:int(want["out_offsets"][-1])]
    want_d = oracle.decode_batch(table, stream, want["out_offsets"], 8 * len(stream) + 16)
    got_d = ctx.decode(stream, want["out_offsets"], 8 * len(stream) + 16)
    assert_same_packed(got_d, want_d)
    n = len(lens)
    caps = np.maximum(0, want["out_lens"].astype(np.int64) + rng.integers(-9, 2, size=n)).astype(np.uint64)
    slots = np.zeros(n, dtype=np.uint64)
    slots[1:] = np.cumsum(caps)[:-1]
    total = int(caps.sum()) + 1
    assert_same_slotted(ctx.encode(data, offs, total, out_offsets=slots, out_caps=caps),
                        oracle.encode_batch(table, 0xFF, data, offs, total, out_offsets=slots, out_caps=caps), slots)
    ctx.close()


def test_packed_output_too_small_is_a_call_level_short_buffer(contexts, pkg):
    ctx = contexts("hpack")
    data = np.frombuffer(b"www.example.com" * 10, dtype=np.uint8)
    offs = np.arange(0, 151, 15, dtype=np.uint64)
    with pytest.raises(pkg.CodecError) as err:
        ctx.encode(data, offs, out_capacity=20)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER


def test_empty_batches_and_empty_items(contexts):
    ctx = contexts("hpack")
    r = ctx.encode(np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64), 16)
    assert int(r["out_offsets"][0]) == 0
    r = ctx.encode(np.zeros(0, dtype=np.uint8), np.zeros(6, dtype=np.uint64), 16)
    assert not r["out_lens"].any() and not r["status"].any() and not r["out_offsets"].any()
    r = ctx.decode(np.zeros(0, dtype=np.uint8), np.zeros(6, dtype=np.uint64), 16)
    assert not r["out_lens"].any() and not r["status"].any()


# ---- shapes that stress the tiled encoder: tile-straddling items, empties, 1-byte items, one long stream ----

def _check_packed_encode_and_roundtrip(ctx, oracle, table, data, offs, eos=0xFF):
    cap_total = 4 * len(data) + 64
    want = oracle.encode_batch(table, eos, data, offs, cap_total)
    got = ctx.encode(data, offs, cap_total)
    assert_same_packed(got, want)
    stream = want["out"][:int(want["out_offsets"][-1])]
    want_d = oracle.decode_batch(table, stream, want["out_offsets"], len(data) + 64)
    got_d = ctx.decode(stream, want["out_offsets"], len(data) + 64)
    assert_same_packed(got_d, want_d)
    return want


@pytest.mark.parametrize("table_name", ["test", "hpack"])
def test_ragged_item_shapes(contexts, oracle, oracle_tables, table_name):
    rng = np.random.default_rng(0x7117)
    ctx, table = contexts(table_name), oracle_tables[table_name]
    shapes = {
        "mixed": np.concatenate([rng.integers(0, 40, 3000), [4096, 4095, 4097, 1, 0, 0, 12289, 16, 15, 17],
                                 rng.integers(0, 9000, 40), np.zeros(50, dtype=np.int64), [1] * 300, [0, 0, 0]]),
        "all_empty_but_one": np.concatenate([np.zeros(500, dtype=np.int64), [7], np.zeros(500, dtype=np.int64)]),
        "single_bytes": np.ones(9000, dtype=np.int64),
        "tile_multiples": np.array([4096, 8192, 4096, 0, 4096], dtype=np.int64),
        "one_item_exact_tile": np.array([4096], dtype=np.int64),
        "two_items": np.array([5000, 3], dtype=np.int64),
    }
    for name, lens in shapes.items():
        lens = np.asarray(lens, dtype=np.int64)
        if name == "mixed":
            lens = lens[rng.permutation(len(lens))]
        offs = np.zeros(len(lens) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum(lens)
        for zipf in (True, False):
            if zipf:
                data = refcodec.zipf_symbol_sampler(refcodec.table_arrays(table_name)[1])[
                    rng.integers(0, 65536, size=int(offs[-1]))]
            else:
                data = rng.integers(0, 256, size=int(offs[-1]), dtype=np.uint8)
            _check_packed_encode_and_roundtrip(ctx, oracle, table, np.ascontiguousarray(data), offs)


@pytest.mark.parametrize("table_name", ["test", "hpack"])
@pytest.mark.parametrize("nbytes", [1, 15, 16, 17, 4095, 4096, 4097, 1 << 20, (3 << 20) + 5])
def test_single_stream(contexts, oracle, oracle_tables, table_name, nbytes):
    """n == 1: the long-stream path (BASELINE configs 3/4 at a size the oracle finishes quickly)."""
    rng = np.random.default_rng(nbytes)
    ctx, table = contexts(table_name, 0x5A), oracle_tables[table_name]
    sampler = refcodec.zipf_symbol_sampler(refcodec.table_arrays(table_name)[1])
    data = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=nbytes)])
    offs = np.array([0, nbytes], dtype=np.uint64)
    _check_packed_encode_and_roundtrip(ctx, oracle, table, data, offs, eos=0x5A)


def test_worst_case_expansion(contexts, oracle, oracle_tables):
    """All-longest-code input (30-bit HPACK codes, 3.75x expansion) and all-shortest-code input."""
    ctx, table = contexts("hpack"), oracle_tables["hpack"]
    for sym, n in ((10, 20000), (ord("0"), 20000), (22, 4096 * 3 + 1)):
        data = np.full(n, sym, dtype=np.uint8)
        for offs in (np.array([0, n], dtype=np.uint64), np.arange(0, n + 1, 1, dtype=np.uint64)[::7].copy()):
            offs = np.ascontiguousarray(np.append(offs[offs < n], n).astype(np.uint64))
            _check_packed_encode_and_roundtrip(ctx, oracle, table, data, offs)


def test_device_pointer_entry_points(contexts, oracle, oracle_tables):
    """aws_huffman_*_batch_device on torch CUDA tensors, including a misaligned input pointer."""
    import torch
    ctx, table = contexts("hpack"), oracle_tables["hpack"]
    rng = np.random.default_rng(77)
    data, offs = refcodec.random_batch(rng, 30000, 0, 200, "hpack")
    want = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
    total = int(want["out_offsets"][-1])
    dev = torch.device("cuda", 0)
    n = len(offs) - 1
    for shift in (0, 3):
        raw = torch.zeros(len(data) + 16, dtype=torch.uint8, device=dev)
        raw[shift:shift + len(data)] = torch.from_numpy(data).to(dev)
        d_in = raw[shift:shift + len(data)]
        d_off = torch.from_numpy(offs.view(np.int64)).to(dev)
        out_buf = torch.zeros(4 * len(data) + 64 + 16, dtype=torch.uint8, device=dev)
        d_out = out_buf[shift:]
        d_out_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        d_lens = torch.zeros(n, dtype=torch.int64, device=dev)
        st = torch.cuda.Stream(dev)
        with torch.cuda.stream(st):
            ctx.encode_device(n, {"in_": d_in, "in_offsets": d_off, "out": d_out, "out_offsets": d_out_off,
                                  "out_lens": d_lens}, len(data), 4 * len(data) + 64, stream=st.cuda_stream)
            st.synchronize()
            assert np.array_equal(d_out_off.cpu().numpy().view(np.uint64), want["out_offsets"])
            assert np.array_equal(d_out[:total].cpu().numpy(), want["out"][:total])
            assert np.array_equal(d_lens.cpu().numpy().view(np.uint64), want["out_lens"])
            back = torch.zeros(len(data) + 64, dtype=torch.uint8, device=dev)
            back_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            ctx.decode_device(n, {"in_": d_out, "in_offsets": d_out_off, "out": back, "out_offsets": back_off},
                              total, len(data) + 64, stream=st.cuda_stream)
            st.synchronize()
            assert np.array_equal(back[:len(data)].cpu().numpy(), data)
            assert np.array_equal(back_off.cpu().numpy().view(np.uint64), offs)


# ---- long single stream: chunked speculative decode -------------------------------------------------------

@pytest.mark.parametrize("table_name", ["test", "hpack"])
def test_single_stream_of_arbitrary_bytes(contexts, oracle, oracle_tables, table_name):
    """Random / corrupted long streams: the true path hits UNKNOWN_SYMBOL somewhere (or ends in padding);
    symbols, status, cursor and leftover register must match the reference loop exactly."""
    rng = np.random.default_rng(0x5EED)
    ctx, table = contexts(table_name), oracle_tables[table_name]
    sampler = refcodec.zipf_symbol_sampler(refcodec.table_arrays(table_name)[1])
    clean = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=600_000)])
    enc = oracle.encode_batch(table, 0xFF, clean, [0, len(clean)], 4 * len(clean) + 64)
    stream = enc["out"][:int(enc["out_offsets"][-1])].copy()
    cases = [stream]
    for where in (len(stream) - 3, len(stream) // 2, 70_000):
        broken = stream.copy()
        broken[where:where + 6] = 0xFF  # 48 one-bits: no code in either table
        cases.append(broken)
    cases.append(rng.integers(0, 256, size=200_000, dtype=np.uint8))
    cases.append(np.concatenate([stream[:100_000], np.zeros(50_000, dtype=np.uint8)]))
    for payload in cases:
        payload = np.ascontiguousarray(payload)
        offs = np.array([0, len(payload)], dtype=np.uint64)
        cap = 2 * len(payload) + 64 if table_name == "hpack" else 2 * len(payload) + 64
        want = oracle.decode_batch(table, payload, offs, cap)
        got = ctx.decode(payload, offs, cap)
        assert_same_packed(got, want)


def test_stream_that_never_self_synchronises(pkg, oracle):
    """A code whose misaligned decodes never find the true boundaries again: symbol 0 has a 4-bit code,
    every other code is 8 bits with two non-zero nibbles. After one 4-bit code the rest of the stream sits
    at bit offset 4 mod 8 and every speculative start is wrong, so the repair path must fix it all."""
    patterns = np.zeros(256, dtype=np.uint32)
    num_bits = np.zeros(256, dtype=np.uint8)
    patterns[0], num_bits[0] = 0x0, 4
    sym = 1
    for hi in range(1, 16):
        for lo in range(1, 16):
            patterns[sym], num_bits[sym] = (hi << 4) | lo, 8
            sym += 1
    table = oracle.table(patterns, num_bits)
    coder = pkg.capi.python_coder(lambda s: (patterns[s], num_bits[s]))
    ctx = pkg.BatchContext(coder, device=0)
    rng = np.random.default_rng(4)
    for n in (70_000, 200_001):
        data = rng.integers(1, 226, size=n).astype(np.uint8)
        data[0] = 0
        data[n // 3] = 0  # shifts alignment back mid-stream
        offs = np.array([0, n], dtype=np.uint64)
        want = oracle.encode_batch(table, 0xFF, data, offs, n + 64)
        got = ctx.encode(data, offs, n + 64)
        assert_same_packed(got, want)
        stream = want["out"][:int(want["out_offsets"][-1])]
        want_d = oracle.decode_batch(table, stream, want["out_offsets"], 2 * n + 64)
        got_d = ctx.decode(stream, want["out_offsets"], 2 * n + 64)
        assert_same_packed(got_d, want_d)
    ctx.close()


def test_pipelined_host_path(contexts, oracle, oracle_tables, pkg):
    """Host entry points with a batch big enough (>= 8 MB) to be cut into overlapping sub-batches: results
    must be identical to one shot, including the call-level SHORT_BUFFER with complete offsets."""
    rng = np.random.default_rng(0x91E)
    ctx, table = contexts("hpack"), oracle_tables["hpack"]
    data, offs = refcodec.random_batch(rng, 300_000, 0, 256, "hpack")
    assert len(data) > 34 << 20
    cap = 2 * len(data)
    want = oracle.encode_batch(table, 0xFF, data, offs, cap)
    got = ctx.encode(data, offs, cap)
    assert_same_packed(got, want)
    total = int(want["out_offsets"][-1])
    stream = want["out"][:total]
    want_d = oracle.decode_batch(table, stream, want["out_offsets"], len(data) + 64)
    got_d = ctx.decode(stream, want["out_offsets"], len(data) + 64)
    assert_same_packed(got_d, want_d)
    lean = ctx.encode(data, offs, cap, extras=False)
    assert np.array_equal(lean["out_offsets"], want["out_offsets"]) and np.array_equal(lean["out"][:total], stream)
    with pytest.raises(pkg.CodecError) as err:
        ctx.encode(data, offs, total - 1)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER


def _pinned(array):
    """A page-locked copy of a numpy array (the host entry points stage it through device memory like any other)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(array)).pin_memory()
    return t.numpy()


@pytest.mark.parametrize("shape", ["batch", "small", "ragged_ends", "stream"])
def test_staged_host_paths_with_pinned_buffers(contexts, oracle, oracle_tables, pkg, shape):
    """Pinned payload buffers of the caller through the staged host paths: one shot ("small", "ragged_ends", "stream")
    and pipelined ("batch" is over 8 MiB). Same results as the oracle, bit for bit; the bytes after the result stay
    untouched."""
    rng = np.random.default_rng({"batch": 1, "small": 2, "ragged_ends": 3, "stream": 4}[shape])
    ctx, table = contexts("hpack"), oracle_tables["hpack"]
    if shape == "batch":
        data, offs = refcodec.random_batch(rng, 120_000, 0, 256, "hpack")
    elif shape == "small":
        data, offs = refcodec.random_batch(rng, 700, 0, 40, "hpack")
    elif shape == "ragged_ends":  # sizes that end right at, or a few bytes off, a 16-byte / page boundary
        data, offs = refcodec.random_batch(rng, 5000, 1, 100, "hpack")
        keep = (len(data) // 4096) * 4096 - 3
        n_keep = int(np.searchsorted(offs, keep, side="right")) - 1
        offs = offs[:n_keep + 1].copy()
        data = data[:int(offs[-1])]
    else:
        data, offs = refcodec.random_batch(rng, 1, 3_000_001, 3_000_001, "hpack")
    cap = 2 * len(data) + 64
    want = oracle.encode_batch(table, 0xFF, data, offs, cap)
    total = int(want["out_offsets"][-1])

    out = _pinned(np.full(cap, 0xA5, dtype=np.uint8))
    got = ctx.encode(_pinned(data), offs, cap, out=out)
    assert_same_packed(got, want)
    assert (got["out"][total:] == 0xA5).all(), "bytes after the result were touched"

    stream = want["out"][:total]
    want_d = oracle.decode_batch(table, stream, want["out_offsets"], len(data) + 64)
    out_d = _pinned(np.full(len(data) + 64, 0x5A, dtype=np.uint8))
    got_d = ctx.decode(_pinned(stream), want["out_offsets"], len(data) + 64, out=out_d)
    assert_same_packed(got_d, want_d)
    assert (got_d["out"][len(data):] == 0x5A).all()

    # the call-level SHORT_BUFFER: offsets complete, nothing past the capacity written
    small = _pinned(np.full(total + 32, 0x77, dtype=np.uint8))
    with pytest.raises(pkg.CodecError) as err:
        ctx.encode(_pinned(data), offs, total - 1, out=small)
    assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
    assert (small[total - 1:] == 0x77).all()


@pytest.mark.parametrize("table_name", ["test", "hpack"])
def test_stream_lengths_around_chunk_boundaries(contexts, oracle, oracle_tables, table_name):
    """The fused stream decoder lets its last 1024-bit chunk absorb a tail of fewer than 32 bits: decode
    streams whose encoded length sits just before / on / just after a chunk boundary, and streams cut at
    an arbitrary byte (the last code is cut short: what remains is 'padding' or an incomplete code)."""
    rng = np.random.default_rng(0xC0FFEE)
    ctx, table = contexts(table_name), oracle_tables[table_name]
    sampler = refcodec.zipf_symbol_sampler(refcodec.table_arrays(table_name)[1])
    data = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=400000)])
    offs = np.array([0, len(data)], dtype=np.uint64)
    enc = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
    stream = enc["out"][:int(enc["out_offsets"][-1])]
    assert len(stream) > 200000
    base = (len(stream) // 128 - 3) * 128  # a multiple of the chunk size (128 bytes)
    for cut in (base - 1, base, base + 1, base + 2, base + 3, base + 4, base + 5, base + 127, 65536, 65537, 131072 + 3):
        part = np.ascontiguousarray(stream[:cut])
        o = np.array([0, cut], dtype=np.uint64)
        want = oracle.decode_batch(table, part, o, len(data) + 64)
        got = ctx.decode(part, o, len(data) + 64)
        assert_same_packed(got, want)


def test_encode_lengths_around_tile_boundaries(contexts, oracle, oracle_tables):
    """Items and streams whose sizes straddle the encoder's 8 KiB tiles and 32-symbol thread ranges."""
    rng = np.random.default_rng(0x71E5)
    ctx, table = contexts("hpack"), oracle_tables["hpack"]
    sampler = refcodec.zipf_symbol_sampler(refcodec.table_arrays("hpack")[1])
    for n in (8191, 8192, 8193, 16384, 16385, 8192 * 3 - 1, 8192 * 5 + 31, 8192 * 5 + 32, 8192 * 5 + 33):
        data = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=n)])
        _check_packed_encode_and_roundtrip(ctx, oracle, table, data, np.array([0, n], dtype=np.uint64))
    # item starts on, just before and just after tile and thread boundaries; runs of empty items between them
    lens = np.array([8192, 0, 0, 1, 8191, 31, 1, 32, 0, 33, 8192 * 2 - 97, 97, 5, 0, 8192, 8192, 3, 0], dtype=np.int64)
    offs = np.zeros(len(lens) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(lens)
    data = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=int(offs[-1]))])
    _check_packed_encode_and_roundtrip(ctx, oracle, table, data, offs)


def test_batch_decode_with_oversized_strings(contexts, oracle, oracle_tables):
    """Tiles of the batch decoder that do not fit its shared-memory stage (a few very long strings among
    short ones) take the two-pass global-memory route; tiles next to them stay on the fast route."""
    rng = np.random.default_rng(0xB16)
    ctx, table = contexts("hpack"), oracle_tables["hpack"]
    sampler = refcodec.zipf_symbol_sampler(refcodec.table_arrays("hpack")[1])
    lens = rng.integers(8, 257, size=2000)
    lens[[5, 700, 701, 1500]] = [40000, 3000, 70000, 2561]
    offs = np.zeros(len(lens) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(lens)
    data = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=int(offs[-1]))])
    _check_packed_encode_and_roundtrip(ctx, oracle, table, data, offs)


@pytest.mark.parametrize("lo,hi", [(200, 256), (600, 900), (1, 6), (2000, 2400)])
def test_batch_decode_string_length_regimes(contexts, oracle, oracle_tables, lo, hi):
    """The batch decoder takes fewer strings per tile when the strings are long (so that a tile of average
    strings still fits its shared-memory stage) and the full 288 when they are short."""
    rng = np.random.default_rng(lo * 7 + hi)
    ctx, table = contexts("hpack"), oracle_tables["hpack"]
    data, offs = refcodec.random_batch(rng, 3000 if hi < 1000 else 700, lo, hi, "hpack")
    _check_packed_encode_and_roundtrip(ctx, oracle, table, data, offs)


def test_context_from_the_generators_code_table(pkg, coders, oracle, oracle_tables):
    """A context built from <name>_get_code_table() (no callbacks) encodes and decodes like the one built
    from <name>_get_coder()."""
    rng = np.random.default_rng(0x7AB1E)
    sampler = refcodec.zipf_symbol_sampler(refcodec.table_arrays("hpack")[1])
    lens = rng.integers(0, 300, size=3000)
    offs = np.zeros(len(lens) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(lens)
    data = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=int(offs[-1]))])
    ctx = pkg.BatchContext(None, eos_padding=0xFF, device=0, code_table=coders.code_table_pointer("hpack"))
    try:
        _check_packed_encode_and_roundtrip(ctx, oracle, oracle_tables["hpack"], data, offs)
    finally:
        ctx.close()
