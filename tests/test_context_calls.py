"""A host-pointer call waits for the device calls of its context that are still in flight on other streams: both kinds
of call share the context's scratch, staging and HPACK buffers. Each case queues a _device call on a side stream
behind a long sleep, makes a host call on the same context, and checks that the device call had finished when the host
call returned and that both results match the oracle."""
import numpy as np
import pytest

import hpack_records_oracle as rec
import refcodec
import test_hpack_header_blocks as base

lit = rec.lit
pytestmark = pytest.mark.gpu

SLEEP_CYCLES = 2_000_000_000  # about a second of spinning ahead of the device call


@pytest.fixture(scope="module")
def ctx(pkg, coders):
    c = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
    yield c
    c.close()


def _dev(a):
    import torch
    a = np.require(a, requirements=["C", "W"])
    return torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a).to("cuda:0")


def _zeros(n, dtype):
    import torch
    return torch.zeros(max(int(n), 1), dtype=dtype, device="cuda:0")


def _host_array(t):
    a = t.cpu().numpy()
    return a.view(np.uint64) if a.dtype == np.int64 else a


def huffman_case(ctx, oracle, oracle_tables):
    """device: aws_huffman_decode_batch_device; host: aws_huffman_encode_batch."""
    import torch
    table = oracle_tables["hpack"]
    rng = np.random.default_rng(31)
    data, offs = refcodec.random_batch(rng, 3000, 0, 200, "hpack")
    enc = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
    total = int(enc["out_offsets"][-1])
    n = len(offs) - 1
    d_in, d_in_off = _dev(enc["out"][:total]), _dev(enc["out_offsets"])
    d_out, d_out_off = _zeros(len(data) + 64, torch.uint8), _zeros(n + 1, torch.int64)

    def device_call(stream):
        ctx.decode_device(n, {"in_": d_in, "in_offsets": d_in_off, "out": d_out, "out_offsets": d_out_off}, total,
                          len(data) + 64, stream=stream)

    def check_device():
        assert np.array_equal(_host_array(d_out_off), offs)
        assert np.array_equal(_host_array(d_out)[:len(data)], data)

    host_data, host_offs = refcodec.random_batch(rng, 3000, 0, 200, "hpack")
    host_want = oracle.encode_batch(table, 0xFF, host_data, host_offs, 4 * len(host_data) + 64)

    def host_call():
        got = ctx.encode(host_data, host_offs, out_capacity=4 * len(host_data) + 64)
        t = int(host_want["out_offsets"][-1])
        assert np.array_equal(got["out_offsets"], host_want["out_offsets"])
        assert np.array_equal(got["out"][:t], host_want["out"][:t])
        assert np.array_equal(got["status"], host_want["status"])

    return device_call, check_device, host_call, (d_out, d_out_off)


def hpack_strings_case(ctx, oracle, oracle_tables):
    """device: aws_hpack_string_decode_batch_device; host: aws_hpack_string_encode_batch."""
    import torch
    lo = lit.LiteralOracle(oracle, oracle_tables["hpack"])
    rng = np.random.default_rng(32)
    data, offs = refcodec.random_batch(rng, 3000, 0, 100, "hpack")
    framed, framed_offs = lo.encode_batch(data, offs, lit.ALWAYS)
    want, want_offs, want_status = lo.decode_batch(framed, framed_offs)
    n = len(offs) - 1
    d_in, d_in_off = _dev(framed), _dev(framed_offs)
    d_out, d_out_off = _zeros(2 * len(data) + 64, torch.uint8), _zeros(n + 1, torch.int64)
    d_status = _zeros(n, torch.int32)

    def device_call(stream):
        ctx.hpack_device(False, n, d_in, d_in_off, len(framed), d_out, d_out.numel(), d_out_off, status=d_status,
                         stream=stream)

    def check_device():
        assert np.array_equal(_host_array(d_status)[:n], want_status)
        assert np.array_equal(_host_array(d_out_off), want_offs)
        assert np.array_equal(_host_array(d_out)[:len(want)], want)

    host_data, host_offs = refcodec.random_batch(rng, 3000, 0, 100, "hpack")
    host_want, host_want_offs = lo.encode_batch(host_data, host_offs, lit.SMALLEST)

    def host_call():
        got = ctx.hpack_encode_strings(host_data, host_offs, out_capacity=len(host_want) + 64, mode=lit.SMALLEST)
        assert np.array_equal(got["out_offsets"], host_want_offs)
        assert np.array_equal(got["out"][:len(host_want)], host_want)

    return device_call, check_device, host_call, (d_out, d_out_off, d_status)


def header_blocks_case(ctx, oracle, oracle_tables):
    """device: aws_hpack_header_block_encode_records_batch_device; host: aws_hpack_header_block_decode_batch."""
    import torch
    block_oracle = rec.RecordsOracle(lit.LiteralOracle(oracle, oracle_tables["hpack"]))
    rng = np.random.default_rng(33)
    lists = rec.records_batch([block_oracle.random_block(rng, base._text)[1] for _ in range(500)])
    want = block_oracle.encode_records_batch(*lists, mode=lit.ALWAYS)
    n, F = len(lists[0]) - 1, int(lists[0][-1])
    fo, kind, index, strings, so = (_dev(a) for a in lists)
    out, out_off = _zeros(len(want[0]) + 64, torch.uint8), _zeros(n + 1, torch.int64)
    status = _zeros(n, torch.int32)

    def device_call(stream):
        ctx.hpack_encode_records_device(n, fo, F, kind, index, strings, so, len(lists[3]), out, out_off, status,
                                        mode=lit.ALWAYS, stream=stream)

    def check_device():
        got_out, got_offs, got_status = _host_array(out), _host_array(out_off), _host_array(status)[:n]
        assert np.array_equal(got_status, want[2])
        assert np.array_equal(got_offs, want[1])
        assert np.array_equal(got_out[:len(want[0])], want[0])

    host_data, host_offs = base._batch([block_oracle.random_block(rng, base._any_bytes)[0] for _ in range(500)])
    host_want = block_oracle.decode_batch(host_data, host_offs)

    def host_call():
        base.assert_decode_matches(ctx.hpack_decode_blocks(host_data, host_offs), host_want)

    return device_call, check_device, host_call, (out, out_off, status)


CASES = {"huffman": huffman_case, "hpack_strings": hpack_strings_case, "header_blocks": header_blocks_case}


@pytest.mark.parametrize("case", sorted(CASES))
def test_host_call_waits_for_device_calls_on_other_streams(ctx, oracle, oracle_tables, case):
    import torch
    device_call, check_device, host_call, outputs = CASES[case](ctx, oracle, oracle_tables)
    side = torch.cuda.Stream()
    device_call(side.cuda_stream)  # warm-up: every buffer of both calls has grown, so neither call synchronises
    host_call()
    torch.cuda.synchronize()
    for t in outputs:
        t.zero_()

    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
    device_call(side.cuda_stream)
    device_done = torch.cuda.Event()
    device_done.record(side)
    host_call()
    finished = device_done.query()
    side.synchronize()
    assert finished, "the host call returned while the device call was still queued on the other stream"
    check_device()
