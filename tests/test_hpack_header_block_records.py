"""HPACK header blocks from field records (aws_hpack_header_block_encode_records_batch[_device],
include/aws/compression/hpack_header_block_batch.h): the encode side of a caller that keeps its own dynamic table.

CPU part (-m "not gpu"): the records oracle (tests/hpack_records_oracle.py) gives back RFC 7541 Appendix C's octets
from the decoder's records; its encoder-side table policy (EncoderTable) reproduces the RFC's own representations;
policy records survive encode -> decode -> the decoder-side table replay on random connections; the header compiles;
no device means no result.
GPU part: the entry points against that oracle, array for array (out, out_offsets, status)."""
import ctypes as C

import numpy as np
import pytest

import hpack_records_oracle as rec
import test_hpack_header_blocks as base

blk, lit = rec.blk, rec.lit
I, INC, WO, NV, SU, AUTO = rec.INDEXED, rec.INCREMENTAL, rec.WITHOUT, rec.NEVER, rec.SIZE_UPDATE, rec.AUTO
RFC = base.RFC7541_BLOCKS


@pytest.fixture(scope="module")
def block_oracle(oracle, oracle_tables):
    return rec.RecordsOracle(lit.LiteralOracle(oracle, oracle_tables["hpack"]))


def rfc_mode(name):
    """C.2, C.3 and C.5 send raw literals, C.4 and C.6 Huffman-coded ones."""
    return lit.ALWAYS if name[:3] in ("C.4", "C.6") else lit.NEVER


def _connection(rng, max_size, n_lists):
    """(table size changes, header lists, never-indexed flags) of one random connection: headers drawn from a small
    pool so that they repeat, long values that force eviction, sizes that change between lists."""
    pool = [(b":method", b"GET"), (b":path", b"/"), (b":authority", b"example.com"), (b"user-agent", b"probe/1.0"),
            (b"cookie", b"a=1; b=2"), (b"x-trace", b"abc"), (b"x-trace", b"def"), (b"accept", b"*/*"),
            (b"", b""), (b"x-empty", b"")]
    sizes, lists, flags = [], [], []
    for _ in range(n_lists):
        sizes.append(int(rng.choice([0, 64, 256, max_size])) if rng.random() < 0.15 else None)
        headers = []
        for _ in range(int(rng.integers(0, 9))):
            r = rng.random()
            if r < 0.6:
                headers.append(pool[int(rng.integers(0, len(pool)))])
            elif r < 0.8:
                headers.append((base._text(rng, int(rng.integers(1, 12))), base._any_bytes(rng, int(rng.integers(0, 30)))))
            else:  # larger than a 256-octet table, or most of it
                headers.append((b"x-big", base._text(rng, int(rng.choice([100, 200, 300])))))
        lists.append(headers)
        flags.append([1 if rng.random() < 0.1 else 0 for _ in headers])
    return sizes, lists, flags


def _policy_records(max_size, sizes, lists, flags):
    table = rec.EncoderTable(max_size)
    out = []
    for size, headers, never in zip(sizes, lists, flags):
        if size is not None:
            table.set_max_size(size)
        out.append(table.records(headers, never))
    return out


def _replay(max_size, blocks_records):
    table = base.DynamicTable(max_size)
    return [table.resolve(records) for records in blocks_records]


# ------------------------------------------------------------------------------------------------ CPU
def test_oracle_records_encode_to_the_rfc_octets(block_oracle):
    for name, (hexed, _) in RFC.items():
        st, records = block_oracle.decode_block(bytes.fromhex(hexed))
        assert st == lit.OK
        assert block_oracle.encode_records(records, mode=rfc_mode(name)) == (lit.OK, bytes.fromhex(hexed)), name


@pytest.mark.parametrize("blocks,max_size,lists,sizes", [
    (["C.3.1", "C.3.2", "C.3.3"], 4096, base.REQUESTS, [57, 110, 164]),
    (["C.5.1", "C.6.2", "C.6.3"], 256, base.RESPONSES, [222, 222, 215]),
])
def test_policy_reproduces_the_rfc_representations(block_oracle, blocks, max_size, lists, sizes):
    """RFC 7541's own encoder indexes every field: the policy's records are the RFC's, and they encode to its octets
    (raw for C.3 / C.5, Huffman for C.4 / C.6)."""
    table = rec.EncoderTable(max_size)
    for name, headers, size in zip(blocks, lists, sizes):
        records = table.records(headers)
        assert records == base.expected_records(RFC[name][1]), name
        assert table.size == size, name
        huffman = {"C.3": "C.4", "C.5": "C.6"}.get(name[:3], name[:3]) + name[3:]
        for rfc_name in {name, huffman}:
            assert block_oracle.encode_records(records, mode=rfc_mode(rfc_name)) == (
                lit.OK, bytes.fromhex(RFC[rfc_name][0])), rfc_name


def test_policy_size_updates_and_eviction():
    table = rec.EncoderTable(256)
    assert table.records([(b"x-a", b"1" * 100)]) == [(INC, 0, b"x-a", b"1" * 100)]
    assert table.records([(b"x-a", b"1" * 100), (b"x-a", b"2")]) == [(I, 62, b"", b""), (INC, 62, b"", b"2")]
    table.set_max_size(64)  # only x-a: 2 (36 octets) stays
    table.set_max_size(128)
    assert table.size == 36 and len(table.entries) == 1
    assert table.records([(b"x-a", b"2")]) == [(SU, 64, b"", b""), (SU, 128, b"", b""), (I, 62, b"", b"")]
    assert table.records([(b"x-b", b"v" * 200)]) == [(INC, 0, b"x-b", b"v" * 200)]  # 235 > 128: empties the table
    assert table.size == 0
    assert table.records([(b"cookie", b"s"), (b"x-a", b"2")], [1, 0]) == [(NV, 32, b"cookie", b"s"),
                                                                        (INC, 0, b"x-a", b"2")]


@pytest.mark.parametrize("max_size", [256, 4096])
def test_policy_records_round_trip_through_the_decoder_table(block_oracle, max_size):
    rng = np.random.default_rng(max_size)
    kinds = set()
    for _ in range(12):
        sizes, lists, flags = _connection(rng, max_size, 25)
        records = _policy_records(max_size, sizes, lists, flags)
        decoded = []
        for recs in records:
            st, octets = block_oracle.encode_records(recs, mode=int(rng.integers(0, 3)))
            assert st == lit.OK
            st, back = block_oracle.decode_block(octets)
            assert (st, back) == (lit.OK, recs)
            decoded.append(back)
            kinds |= {r[0] for r in recs}
        assert _replay(max_size, decoded) == [[(bytes(n), bytes(v)) for n, v in h] for h in lists]
    assert kinds == {I, INC, NV, SU}


def test_oracle_invalid_records(block_oracle):
    enc = block_oracle.encode_records
    good = [(I, 2, b"", b"")]
    assert enc(good) == (lit.OK, b"\x82")
    for bad in ([(6, 1, b"", b"")], [(255, 1, b"", b"")], [(I, 0, b"", b"")], good + [(SU, 0, b"", b"")],
                [(I, 127 + (1 << 63), b"", b"")], [(SU, (1 << 64) - 1, b"", b"")],
                [(INC, 63 + (1 << 63), b"", b"v")]):
        assert enc(bad) == (lit.INVALID_ARGUMENT, b""), bad
    # the largest integers a decoder takes: 9 continuation octets
    for kind, bits in ((I, 7), (INC, 6), (WO, 4), (NV, 4), (SU, 5)):
        top = (1 << bits) - 2 + (1 << 63)
        st, octets = enc([(SU, 0, b"", b"")] + [(kind, top, b"", b"")])
        assert st == lit.OK and len(octets) == 1 + 10 + (kind in (INC, WO, NV))
        assert block_oracle.decode_block(octets)[1][1][:2] == (kind, top)


def test_header_declares_the_records_entry_points(pkg, tmp_path):
    import subprocess
    inc = [a for d in pkg._build.INCLUDES for a in ("-I", d)]
    for compiler, ext, std in (("gcc", "c", "-std=c99"), ("g++", "cpp", "-std=c++14")):
        src = tmp_path / ("records." + ext)
        src.write_text("#include <aws/compression/hpack_header_block_batch.h>\n"
                       "int main(void){enum aws_hpack_field_kind k = AWS_HPACK_FIELD_AUTO;\n"
                       "int (*h)(struct aws_huffman_batch_ctx *, const struct aws_hpack_header_lists *,\n"
                       "  enum aws_hpack_huffman_mode, uint8_t *, uint64_t, uint64_t *, int32_t *) =\n"
                       "  aws_hpack_header_block_encode_records_batch;\n"
                       "int (*d)(struct aws_huffman_batch_ctx *, const struct aws_hpack_header_lists *, uint64_t,\n"
                       "  uint64_t, enum aws_hpack_huffman_mode, uint8_t *, uint64_t, uint64_t *, int32_t *, void *) =\n"
                       "  aws_hpack_header_block_encode_records_batch_device;\n"
                       "(void)k; (void)h; (void)d; return k == 5 ? 0 : 1;}\n")
        subprocess.check_call([compiler, std, "-Wall", "-Werror", *inc, "-c", "-o", str(tmp_path / "o.o"), str(src)])


def test_no_device_means_no_result(pkg, coders, product):
    """Without a device there is no context (AWS_ERROR_COMPRESSION_DEVICE_FAILURE), and the records entry points
    without a context fail with AWS_ERROR_INVALID_ARGUMENT and write nothing, like the other entry points."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.CodecError) as err:
        pkg.BatchContext(coders.coder("hpack"), device=0)
    assert err.value.code == pkg.AWS_ERROR_COMPRESSION_DEVICE_FAILURE
    L = product.lib
    fo, so = np.array([0, 1], np.uint64), np.array([0, 0, 0], np.uint64)
    kind, index = np.array([I], np.uint8), np.array([2], np.uint64)
    lists = pkg.capi.aws_hpack_header_lists(1, fo.ctypes.data, 0, kind.ctypes.data, index.ctypes.data, None, None, 0,
                                            so.ctypes.data)
    out, offs, status = np.zeros(8, np.uint8), np.full(2, 7, np.uint64), np.full(1, 7, np.int32)
    for call in (lambda: L.aws_hpack_header_block_encode_records_batch(
                     None, C.byref(lists), 0, out.ctypes.data, 8, offs.ctypes.data, status.ctypes.data),
                 lambda: L.aws_hpack_header_block_encode_records_batch_device(
                     None, C.byref(lists), 1, 0, 0, out.ctypes.data, 8, offs.ctypes.data, status.ctypes.data, None)):
        L.aws_reset_error()
        assert call() == pkg.capi.AWS_OP_ERR
        assert L.aws_last_error() == pkg.capi.AWS_ERROR_INVALID_ARGUMENT
    assert (offs == 7).all() and (status == 7).all() and not out.any()


# ------------------------------------------------------------------------------------------------ GPU
hpack_ctx = base.hpack_ctx


def _blocks_of(data, offs):
    return [bytes(data[int(offs[i]):int(offs[i + 1])]) for i in range(len(offs) - 1)]


def _decoded_records(got):
    """The record lists of a decode result, per block."""
    fo, so, strings = got["field_offsets"], got["string_offsets"], got["strings"]
    return [[(int(got["field_kind"][f]), int(got["field_index"][f]),
              bytes(strings[int(so[2 * f]):int(so[2 * f + 1])]), bytes(strings[int(so[2 * f + 1]):int(so[2 * f + 2])]))
             for f in range(int(fo[b]), int(fo[b + 1]))] for b in range(len(fo) - 1)]


def _to_dev(*arrays):
    import torch
    arrays = [np.require(a, requirements=["C", "W"]) for a in arrays]
    return [torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a).to("cuda:0") for a in arrays]


def _encode_records_device(ctx, lists, mode, out_capacity, never=None, stream=None):
    """records_batch arrays through the _device entry point; returns (out, out_offsets, status) on the host."""
    import torch
    fo, kind, index, strings, so = lists
    n, F = len(fo) - 1, int(fo[-1])
    d_fo, d_kind, d_index, d_strings, d_so = _to_dev(fo, kind, index, strings, so)
    d_never = _to_dev(never)[0] if never is not None else None
    out = torch.zeros(out_capacity + 64, dtype=torch.uint8, device="cuda:0")
    out_off = torch.zeros(n + 1, dtype=torch.int64, device="cuda:0")
    status = torch.full((n,), -1, dtype=torch.int32, device="cuda:0")
    ctx.hpack_encode_records_device(n, d_fo, F, d_kind, d_index, d_strings, d_so, len(strings), out, out_off, status,
                                    mode=mode, never_indexed=d_never, out_capacity=out_capacity, stream=stream)
    torch.cuda.synchronize()
    return out.cpu().numpy(), out_off.cpu().numpy().view(np.uint64), status.cpu().numpy()


def _decode_device(ctx, data, offs):
    import torch
    n, size = len(offs) - 1, int(offs[-1])
    d_in, d_off = _to_dev(data, offs)
    r = {"field_offsets": torch.zeros(n + 1, dtype=torch.int64, device="cuda:0"),
         "field_kind": torch.zeros(size + 1, dtype=torch.uint8, device="cuda:0"),
         "field_index": torch.zeros(size + 1, dtype=torch.int64, device="cuda:0"),
         "strings": torch.zeros(28 * size + 1, dtype=torch.uint8, device="cuda:0"),
         "string_offsets": torch.zeros(2 * size + 1, dtype=torch.int64, device="cuda:0"),
         "status": torch.full((n,), -1, dtype=torch.int32, device="cuda:0")}
    ctx.hpack_decode_blocks_device(n, d_in, d_off, size, r["field_offsets"], r["field_kind"], r["field_index"],
                                   r["strings"], r["string_offsets"], status=r["status"])
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy() for k, v in r.items()}
    for k in ("field_offsets", "field_index", "string_offsets"):
        got[k] = got[k].view(np.uint64)
    return got


def assert_encode_matches(got, want):
    out, offs, status = got
    w_out, w_offs, w_status = want
    assert np.array_equal(status, w_status), np.flatnonzero(status != w_status)[:10]
    assert np.array_equal(offs, w_offs)
    assert np.array_equal(out[:len(w_out)], w_out)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["one_kernel", "passes"])
def test_appendix_c_decoded_on_device_encodes_back_to_the_rfc_octets(hpack_ctx, block_oracle, monkeypatch, route):
    if route == "passes":
        monkeypatch.setenv("AWS_HUFFMAN_HPACK_PASSES", "1")
    names = list(RFC)
    data, offs = base._batch([bytes.fromhex(RFC[k][0]) for k in names])
    got = _decode_device(hpack_ctx, data, offs)
    assert not got["status"].any()
    nf = int(got["field_offsets"][-1])
    records = (got["field_offsets"], got["field_kind"][:nf], got["field_index"][:nf],
               got["strings"][:int(got["string_offsets"][2 * nf])], got["string_offsets"][:2 * nf + 1])
    for mode in (lit.NEVER, lit.ALWAYS):
        enc = _encode_records_device(hpack_ctx, records, mode, 4096)
        assert_encode_matches(enc, block_oracle.encode_records_batch(*records, mode=mode))
        assert not enc[2].any()
        for name, octets in zip(names, _blocks_of(*enc[:2])):
            if rfc_mode(name) == mode:
                assert octets == bytes.fromhex(RFC[name][0]), name


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.SMALLEST, lit.NEVER, lit.ALWAYS])
def test_random_blocks_decode_and_encode_back(hpack_ctx, block_oracle, mode):
    rng = np.random.default_rng(70 + mode)
    blocks = [block_oracle.random_block(rng, base._any_bytes, long_values=(200, 600, 30000), mode=mode)[0]
              for _ in range(1200)] + [b""]
    rng.shuffle(blocks)
    data, offs = base._batch(blocks)
    got = hpack_ctx.hpack_decode_blocks(data, offs)
    assert not got["status"].any()
    nf = int(got["field_offsets"][-1])
    kinds, index = got["field_kind"][:nf], got["field_index"][:nf]
    strings, so = got["strings"][:int(got["string_offsets"][2 * nf])], got["string_offsets"][:2 * nf + 1]
    assert set(kinds) == {I, INC, WO, NV, SU}
    assert {62, 127, 128, 300, 70000} <= set(index[kinds == I].tolist()) and (index[kinds == SU] == 1 << 20).any()
    values = [r[3] for recs in _decoded_records(got) for r in recs if r[0] in (INC, WO, NV)]
    assert {2, 3, 4} <= {lit.decode_integer(block_oracle.lit.encode(v, mode), 7)[1] for v in values}
    assert b"" in values
    # the records give back the same octets
    enc = hpack_ctx.hpack_encode_records(got["field_offsets"], kinds, index, strings, so, out_capacity=len(data) + 64,
                                         mode=mode)
    assert not enc["status"].any() and np.array_equal(enc["out_offsets"], offs)
    assert np.array_equal(enc["out"][:len(data)], data)
    # some fields left to the stateless rules (with their never-indexed flags): the oracle on the same records
    auto = rng.random(nf) < 0.3
    kinds2 = np.where(auto & (kinds != SU), AUTO, kinds).astype(np.uint8)
    never = (rng.random(nf) < 0.3).astype(np.uint8)
    want = block_oracle.encode_records_batch(got["field_offsets"], kinds2, index, strings, so, never, mode)
    assert not want[2].any()
    enc = hpack_ctx.hpack_encode_records(got["field_offsets"], kinds2, index, strings, so, out_capacity=len(want[0]) + 64,
                                         mode=mode, never_indexed=never)
    assert_encode_matches((enc["out"], enc["out_offsets"], enc["status"]), want)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [lit.SMALLEST, lit.NEVER, lit.ALWAYS])
def test_auto_records_match_the_stateless_encoder(hpack_ctx, mode):
    rng = np.random.default_rng(50 + mode)  # the lists of test_encode_matches_oracle_and_decodes_back
    fo, strings, so, never = base._random_lists(rng, 800)
    F = len(never)
    want = hpack_ctx.hpack_encode_blocks(fo, strings, so, out_capacity=4 * len(strings) + 16 * F + 64, mode=mode,
                                         never_indexed=never)
    total = int(want["out_offsets"][-1])
    garbage = rng.integers(0, 1 << 40, F).astype(np.uint64)  # the index of an AUTO field is ignored
    got = hpack_ctx.hpack_encode_records(fo, np.full(F, AUTO, np.uint8), garbage, strings, so, out_capacity=total + 64,
                                         mode=mode, never_indexed=never)
    assert not got["status"].any()
    assert np.array_equal(got["out_offsets"], want["out_offsets"])
    assert np.array_equal(got["out"][:total], want["out"][:total])


def _invalid_cases():
    big = 127 + (1 << 63)  # ten continuation octets under the 7-bit prefix
    return [
        [(6, 1, b"", b"")],
        [(I, 2, b"", b""), (255, 0, b"n", b"v")],
        [(I, 0, b"", b"")],
        [(SU, 100, b"", b""), (I, 2, b"", b""), (SU, 4096, b"", b"")],
        [(I, 2, b"", b""), (INC, 0, b"x-n", b"v"), (I, big, b"", b"")],
        [(SU, (1 << 64) - 1, b"", b"")],
        [(WO, 15 + (1 << 63), b"", b"v")],
    ]


@pytest.mark.gpu
def test_invalid_records_give_their_block_nothing(hpack_ctx, block_oracle):
    good = [[(SU, 0, b"", b""), (SU, 4096, b"", b""), (I, 2, b"", b""), (INC, 0, b"custom-key", b"custom-value")],
            [(I, 126 + (1 << 63), b"", b""), (NV, 14 + (1 << 63), b"", b"s"), (INC, 62, b"", b"x")],
            [], [(WO, 4, b":path", b"/sample/path")]]
    blocks = []
    for j, bad in enumerate(_invalid_cases()):
        blocks += [good[j % len(good)], bad]
    blocks += good
    lists = rec.records_batch(blocks)
    want = block_oracle.encode_records_batch(*lists, mode=lit.NEVER)
    bad_blocks = np.arange(1, 2 * len(_invalid_cases()), 2)
    assert (want[2][bad_blocks] == lit.INVALID_ARGUMENT).all() and np.count_nonzero(want[2]) == len(bad_blocks)
    got = hpack_ctx.hpack_encode_records(*lists, out_capacity=len(want[0]) + 64, mode=lit.NEVER)
    assert_encode_matches((got["out"], got["out_offsets"], got["status"]), want)
    sizes = np.diff(got["out_offsets"].astype(np.int64))
    assert (sizes[bad_blocks] == 0).all()
    # the neighbours are the octets of the good blocks alone, and decode back to their records
    alone = rec.records_batch(good)
    ref = hpack_ctx.hpack_encode_records(*alone, out_capacity=4096, mode=lit.NEVER)
    ref_blocks = _blocks_of(ref["out"], ref["out_offsets"])
    got_blocks = _blocks_of(got["out"], got["out_offsets"])
    assert [got_blocks[2 * j] for j in range(len(bad_blocks))] == [ref_blocks[j % len(good)] for j in range(len(bad_blocks))]
    assert got_blocks[-len(good):] == ref_blocks
    back = hpack_ctx.hpack_decode_blocks(ref["out"], ref["out_offsets"])
    assert not back["status"].any() and _decoded_records(back) == [
        [(k, i) + blk.field_strings(k, i, n, v) for k, i, n, v in recs] for recs in good]
    # the device entry point: the same arrays
    dev = _encode_records_device(hpack_ctx, lists, lit.NEVER, len(want[0]) + 64)
    assert_encode_matches(dev, want)


@pytest.mark.gpu
def test_interleaved_connections_end_to_end(hpack_ctx, block_oracle):
    """Several connections, each with its own table, their blocks interleaved in one device batch: device encode,
    device decode, and each connection's replay in block order gives its header lists back."""
    rng = np.random.default_rng(90)
    conns = []
    for c in range(6):
        max_size = (256, 4096)[c % 2]
        sizes, lists, flags = _connection(rng, max_size, 40)
        conns.append((max_size, lists, _policy_records(max_size, sizes, lists, flags)))
    order = [c for c in range(len(conns)) for _ in range(40)]
    rng.shuffle(order)
    taken, blocks, owner = [0] * len(conns), [], []
    for c in order:
        blocks.append(conns[c][2][taken[c]])
        owner.append(c)
        taken[c] += 1
    lists = rec.records_batch(blocks)
    for mode in (lit.SMALLEST, lit.ALWAYS):
        want = block_oracle.encode_records_batch(*lists, mode=mode)
        got = _encode_records_device(hpack_ctx, lists, mode, len(want[0]) + 64)
        assert_encode_matches(got, want)
        back = _decode_device(hpack_ctx, got[0][:len(want[0])], got[1])
        assert not back["status"].any()
        per_block = _decoded_records(back)
        assert per_block == blocks
        for c, (max_size, headers, _) in enumerate(conns):
            mine = [per_block[i] for i in range(len(blocks)) if owner[i] == c]
            assert _replay(max_size, mine) == [[(bytes(n), bytes(v)) for n, v in h] for h in headers], c


@pytest.mark.gpu
def test_capacity_and_arguments(hpack_ctx, block_oracle, pkg):
    rng = np.random.default_rng(5)
    blocks = [block_oracle.random_block(rng, base._text)[1] for _ in range(300)] + _invalid_cases()
    lists = rec.records_batch(blocks)
    want = block_oracle.encode_records_batch(*lists, mode=lit.SMALLEST)
    total = len(want[0])
    assert total > 1000 and want[2].any()
    for cap in (0, 1, total // 2, total - 1):
        with pytest.raises(pkg.CodecError) as err:
            hpack_ctx.hpack_encode_records(*lists, out_capacity=cap)
        assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
        assert np.array_equal(err.value.result["out_offsets"], want[1])
        assert np.array_equal(err.value.result["status"], want[2])
        # device pointers: nothing at or after out_capacity (guard octets behind it)
        import torch
        fo, kind, index, strings, so = _to_dev(*lists)
        out = torch.full((cap + 4096,), 0xA5, dtype=torch.uint8, device="cuda:0")
        out_off = torch.zeros(len(lists[0]), dtype=torch.int64, device="cuda:0")
        status = torch.full((len(blocks),), -1, dtype=torch.int32, device="cuda:0")
        hpack_ctx.hpack_encode_records_device(len(blocks), fo, int(lists[0][-1]), kind, index, strings, so,
                                              len(lists[3]), out, out_off, status, out_capacity=cap)
        torch.cuda.synchronize()
        host = out.cpu().numpy()
        assert (host[cap:] == 0xA5).all()
        assert np.array_equal(host[:cap], want[0][:cap])
        assert np.array_equal(out_off.cpu().numpy().view(np.uint64), want[1])
        assert np.array_equal(status.cpu().numpy(), want[2])
    assert_encode_matches(tuple(hpack_ctx.hpack_encode_records(*lists, out_capacity=total).values()), want)
    # empty batches and lists without fields
    empty = hpack_ctx.hpack_encode_records(np.zeros(1, np.uint64), np.zeros(0, np.uint8), np.zeros(0, np.uint64),
                                           np.zeros(0, np.uint8), np.zeros(1, np.uint64), out_capacity=0)
    assert list(empty["out_offsets"]) == [0]
    none = hpack_ctx.hpack_encode_records(np.zeros(4, np.uint64), np.zeros(0, np.uint8), np.zeros(0, np.uint64),
                                          np.zeros(0, np.uint8), np.zeros(1, np.uint64), out_capacity=0)
    assert list(none["out_offsets"]) == [0] * 4 and list(none["status"]) == [0] * 3
    # the host entry point's checks: NULL kinds or indices, offsets that decrease or do not start at 0
    L = hpack_ctx.library.lib
    fo, kind, index, strings, so = lists
    out, offs, st = np.zeros(16, np.uint8), np.zeros(len(fo), np.uint64), np.zeros(len(blocks), np.int32)

    def call(fo=fo, kind=kind, index=index, so=so):
        h = pkg.capi.aws_hpack_header_lists(len(fo) - 1, fo.ctypes.data, 0, None if kind is None else kind.ctypes.data,
                                            None if index is None else index.ctypes.data, None, strings.ctypes.data, 0,
                                            so.ctypes.data)
        L.aws_reset_error()
        rc = L.aws_hpack_header_block_encode_records_batch(hpack_ctx.handle, C.byref(h), 0, out.ctypes.data, 16,
                                                           offs.ctypes.data, st.ctypes.data)
        return rc, L.aws_last_error()

    bad_fo = fo.copy()
    bad_fo[3], bad_fo[4] = bad_fo[4], bad_fo[3] - 1
    bad_so = so.copy()
    bad_so[0] = 1
    for kw in ({"kind": None}, {"index": None}, {"fo": bad_fo}, {"so": bad_so}, {"fo": fo + 1}):
        assert call(**kw) == (pkg.capi.AWS_OP_ERR, pkg.capi.AWS_ERROR_INVALID_ARGUMENT), kw
    h = pkg.capi.aws_hpack_header_lists(len(fo) - 1, fo.ctypes.data, 0, kind.ctypes.data, None, None, strings.ctypes.data,
                                        0, so.ctypes.data)
    assert L.aws_hpack_header_block_encode_records_batch_device(
        hpack_ctx.handle, C.byref(h), 0, 0, 0, None, 0, offs.ctypes.data, None, None) == pkg.capi.AWS_OP_ERR
    assert L.aws_last_error() == pkg.capi.AWS_ERROR_INVALID_ARGUMENT


@pytest.mark.gpu
def test_device_call_only_enqueues(hpack_ctx, block_oracle):
    """The call returns while a kernel enqueued before it on the same stream still runs: it waited for nothing.
    Then the stream's results match the oracle."""
    import torch
    rng = np.random.default_rng(11)
    lists = rec.records_batch([block_oracle.random_block(rng, base._text)[1] for _ in range(500)])
    want = block_oracle.encode_records_batch(*lists, mode=lit.ALWAYS)
    n, F = len(lists[0]) - 1, int(lists[0][-1])
    fo, kind, index, strings, so = _to_dev(*lists)
    out = torch.zeros(len(want[0]) + 64, dtype=torch.uint8, device="cuda:0")
    out_off = torch.zeros(n + 1, dtype=torch.int64, device="cuda:0")
    status = torch.full((n,), -1, dtype=torch.int32, device="cuda:0")
    stream = torch.cuda.Stream()
    args = (n, fo, F, kind, index, strings, so, len(lists[3]), out, out_off, status)
    hpack_ctx.hpack_encode_records_device(*args, mode=lit.ALWAYS, stream=stream.cuda_stream)  # warm-up: buffers grown
    torch.cuda.synchronize()
    out.zero_()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        torch.cuda._sleep(4_000_000_000)  # about two seconds of spinning ahead of the call
        hpack_ctx.hpack_encode_records_device(*args, mode=lit.ALWAYS, stream=stream.cuda_stream)
        still_running = not stream.query()
    stream.synchronize()
    assert still_running
    assert_encode_matches((out.cpu().numpy(), out_off.cpu().numpy().view(np.uint64), status.cpu().numpy()), want)
