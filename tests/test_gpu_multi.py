"""GPU parity of what round 2 added around the kernels: one batch over several contexts (the multi-GPU split of
BASELINE configs[4], with real kernels on every shard), the pipelined host path with one item larger than a
sub-batch, device-side encoded lengths, a batch beyond 2^31 bytes, and short seeded runs of the fuzz drivers
(the reference's three fuzz properties, tests/fuzz/*.c: encode/decode round trip, decode of arbitrary bytes,
chunked vs one-shot — here as differential runs against the oracle)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import refcodec

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def two_contexts(pkg, coders):
    ctxs = [pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0) for _ in range(2)]
    yield ctxs
    for c in ctxs:
        c.close()


def _same_packed(got, want):
    for k in ("out_offsets", "out_lens", "status", "consumed"):
        assert np.array_equal(got[k], want[k]), k
    total = int(want["out_offsets"][-1])
    assert np.array_equal(got["out"][:total], want["out"][:total])


def test_one_batch_over_two_contexts(pkg, two_contexts, oracle, oracle_tables):
    """aws_huffman_{encode,decode}_batch_multi: plan by bytes -> one context per shard (real kernels) -> host
    concatenation, against the oracle on the whole batch."""
    rng = np.random.default_rng(20260217)
    data, offs = refcodec.random_batch(rng, 40000, 0, 300, "hpack")
    want = oracle.encode_batch(oracle_tables["hpack"], 0xFF, data, offs, 4 * len(data) + 64)
    got = pkg.capi.run_multi(two_contexts, True, data, offs, 4 * len(data) + 64)
    _same_packed(got, want)
    total = int(want["out_offsets"][-1])
    back = pkg.capi.run_multi(two_contexts, False, want["out"][:total], want["out_offsets"], len(data) + 64)
    want_dec = oracle.decode_batch(oracle_tables["hpack"], want["out"][:total], want["out_offsets"], len(data) + 64)
    _same_packed(back, want_dec)
    assert np.array_equal(back["out"][:len(data)], data)


def test_plan_two_contexts_concat_equals_one_shot(pkg, product, two_contexts):
    """The split north_star names, step by step with the public helpers: plan_shards -> shard r on context r ->
    concat_offsets, compared with ONE call on one context."""
    rng = np.random.default_rng(7)
    data, offs = refcodec.random_batch(rng, 30000, 1, 256, "hpack")
    whole = two_contexts[0].encode(data, offs, 4 * len(data) + 64)
    begin = product.plan_shards(offs, 2)
    parts = []
    for r in range(2):
        a, b = int(begin[r]), int(begin[r + 1])
        lo = (offs[a:b + 1] - offs[a]).astype(np.uint64)
        ld = data[int(offs[a]):int(offs[b])]
        parts.append(two_contexts[r].encode(ld, lo, 4 * len(ld) + 64))
    glob = product.concat_offsets([p["out_offsets"] for p in parts])
    assert np.array_equal(glob, whole["out_offsets"])
    payload = np.concatenate([p["out"][:int(p["out_offsets"][-1])] for p in parts])
    assert np.array_equal(payload, whole["out"][:int(whole["out_offsets"][-1])])
    sizes = [int(offs[begin[r + 1]] - offs[begin[r]]) for r in range(2)]
    assert abs(sizes[0] - sizes[1]) <= 512


def test_pipelined_host_path_with_one_item_larger_than_a_sub_batch(pkg, coders, oracle, oracle_tables):
    """Several byte targets of the sub-batch plan fall inside one item: plan_shards returns empty ranges, which the
    pipelined host path must skip (round-1 advisor finding: stale offsets from an empty sub-batch)."""
    rng = np.random.default_rng(99)
    sampler = refcodec.zipf_symbol_sampler(refcodec.table_arrays("hpack")[1])
    small = rng.integers(8, 200, size=60000)
    lens = np.concatenate([small[:30000], [13_000_000], small[30000:]]).astype(np.int64)
    offs = np.zeros(len(lens) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(lens)
    data = sampler[rng.integers(0, 65536, size=int(offs[-1]))]
    assert int(offs[-1]) >= 16 << 20
    ctx = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
    try:
        want = oracle.encode_batch(oracle_tables["hpack"], 0xFF, data, offs, 4 * len(data) + 64)
        got = ctx.encode(data, offs, 4 * len(data) + 64)
        _same_packed(got, want)
        total = int(want["out_offsets"][-1])
        back = ctx.decode(want["out"][:total], want["out_offsets"], len(data) + 64)
        assert np.array_equal(back["out_offsets"], offs)
        assert np.array_equal(back["out"][:len(data)], data)
        assert not back["status"].any()
    finally:
        ctx.close()


def test_encoded_lengths_with_device_pointers(two_contexts, oracle, oracle_tables):
    import torch
    rng = np.random.default_rng(5)
    data, offs = refcodec.random_batch(rng, 5000, 0, 400, "hpack")
    want = oracle.encode_batch(oracle_tables["hpack"], 0xFF, data, offs, 4 * len(data) + 64)["out_lens"]
    d = torch.from_numpy(data).cuda()
    o = torch.from_numpy(offs.astype(np.int64)).cuda()
    lens = torch.zeros(len(offs) - 1, dtype=torch.int64, device="cuda")
    two_contexts[0].encoded_lengths_device(len(offs) - 1, d, o, lens)
    torch.cuda.synchronize()
    assert np.array_equal(lens.cpu().numpy().astype(np.uint64), want)


def test_batch_beyond_two_gib(pkg, coders, oracle, oracle_tables):
    """17.5 M strings, 2.3 GB of symbols generated on the device: byte offsets pass 2^31 (bit positions 2^34).
    GPU bytes and offsets of 4,000 sampled strings against the oracle; decode round trip on the device."""
    import torch
    import bench
    dev = torch.device("cuda", 0)
    free, _ = torch.cuda.mem_get_info()
    if free < 16 << 30:
        pytest.skip("needs 16 GB of free device memory")
    n = 17_500_000
    sampler_np = refcodec.zipf_symbol_sampler(refcodec.table_arrays("hpack")[1])
    sampler_t = torch.from_numpy(sampler_np).to(dev)
    lens = bench.string_lengths_torch(bench.SEED_BATCH, 0, n, dev)
    in_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    in_off[1:] = torch.cumsum(lens, 0)
    raw_bytes = int(in_off[-1].item())
    assert raw_bytes > (1 << 31)
    raw = bench.symbols_torch(bench.SEED_BATCH, 0, raw_bytes, sampler_t, dev)
    cap = raw_bytes + raw_bytes // 2
    enc = torch.empty(cap, dtype=torch.uint8, device=dev)
    enc_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    status = torch.zeros(n, dtype=torch.int32, device=dev)
    ctx = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
    try:
        ctx.encode_device(n, {"in_": raw, "in_offsets": in_off, "out": enc, "out_offsets": enc_off, "status": status},
                          raw_bytes, cap)
        torch.cuda.synchronize()
        assert int(status.abs().sum().item()) == 0
        rng = np.random.default_rng(3)
        picks = np.unique(np.concatenate([rng.integers(0, n, size=3990), [0, 1, n - 2, n - 1], np.arange(n // 2, n // 2 + 6)]))
        idx = torch.from_numpy(picks).to(dev)
        a_in, b_in = in_off[idx].cpu().numpy(), in_off[idx + 1].cpu().numpy()
        a_out, b_out = enc_off[idx].cpu().numpy(), enc_off[idx + 1].cpu().numpy()
        for i in range(len(picks)):
            item = raw[int(a_in[i]):int(b_in[i])].cpu().numpy()
            want = oracle.encode_batch(oracle_tables["hpack"], 0xFF, item, np.array([0, len(item)], dtype=np.uint64), 4 * len(item) + 16)
            wl = int(want["out_offsets"][-1])
            assert int(b_out[i] - a_out[i]) == wl, "encoded length of item %d" % picks[i]
            got = enc[int(a_out[i]):int(b_out[i])].cpu().numpy()
            assert np.array_equal(got, want["out"][:wl]), "bytes of item %d (output offset %d)" % (picks[i], a_out[i])
        enc_bytes = int(enc_off[-1].item())
        assert enc_bytes > (1 << 30)
        dec = torch.empty(raw_bytes + 1024, dtype=torch.uint8, device=dev)
        dec_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        ctx.decode_device(n, {"in_": enc, "in_offsets": enc_off, "out": dec, "out_offsets": dec_off, "status": status},
                          enc_bytes, raw_bytes + 1024)
        torch.cuda.synchronize()
        assert int(status.abs().sum().item()) == 0
        assert torch.equal(dec_off, in_off)
        assert torch.equal(dec[:raw_bytes], raw)
    finally:
        ctx.close()


@pytest.mark.parametrize("script,args", [("fuzz_gpu_codec.py", ["12", "20260217"]), ("fuzz_gpu_literals.py", ["8", "20260217"])])
def test_seeded_fuzz_runs(script, args):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "tests", script)] + args, capture_output=True, text=True,
                          timeout=600)
    assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-2000:]
    print(proc.stdout.strip().splitlines()[-1])


def test_batch_decoder_matches_the_oracle(pkg, coders, oracle, oracle_tables):
    """The batch decoder of the host entry point (decode_batch_kernel) against the oracle: ragged lengths incl. empty,
    very short and long strings, corrupted bytes (unknown symbols, bad padding), both tables, every per-item output
    array."""
    rng = np.random.default_rng(777)
    for table in ("hpack", "test"):
        ctx = pkg.BatchContext(coders.coder(table), eos_padding=0xFF, device=0)
        try:
            for shape in range(5):
                n = int(rng.integers(1, 5000))
                lens = [rng.integers(0, 300, size=n), rng.integers(0, 12, size=n), rng.integers(200, 3000, size=n),
                        np.where(rng.random(n) < 0.3, 0, rng.integers(1, 600, size=n)), rng.integers(1, 40, size=n)][shape]
                offs = np.zeros(n + 1, dtype=np.uint64)
                offs[1:] = np.cumsum(lens)
                sampler = refcodec.zipf_symbol_sampler(refcodec.table_arrays(table)[1])
                data = sampler[rng.integers(0, 65536, size=int(offs[-1]))]
                enc = oracle.encode_batch(oracle_tables[table], 0xFF, data, offs, 4 * len(data) + 64)
                total = int(enc["out_offsets"][-1])
                payload = enc["out"][:total].copy()
                if shape % 2 and total:
                    hits = rng.integers(0, total, size=max(1, total // 400))
                    payload[hits] ^= rng.integers(1, 256, size=len(hits)).astype(np.uint8)
                want = oracle.decode_batch(oracle_tables[table], payload, enc["out_offsets"], 8 * total + 64)
                got = ctx.decode(payload, enc["out_offsets"], 8 * total + 64)
                for k in ("out_offsets", "out_lens", "status", "consumed", "leftover_working_bits", "leftover_num_bits"):
                    assert np.array_equal(got[k], want[k]), (table, shape, k)
                produced = int(want["out_offsets"][-1])
                assert np.array_equal(got["out"][:produced], want["out"][:produced]), (table, shape)
        finally:
            ctx.close()


def test_pipelined_host_path_into_pinned_output(pkg, coders, oracle, oracle_tables):
    """The host entry points with a PINNED output buffer take the pipelined host path (the batch is over 40 MB): the
    sub-batches' payloads are copied into the caller's buffer one after the other. Same bytes, offsets and per-item
    arrays as the oracle — with an odd base address of the buffer, all optional arrays, both directions, and the
    call-level SHORT_BUFFER (offsets complete, payload of the sub-batches that fit still in place)."""
    import torch
    rng = np.random.default_rng(31337)
    ctx = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
    try:
        data, offs = refcodec.random_batch(rng, 400_000, 0, 256, "hpack")
        assert len(data) > 40 << 20
        cap = 2 * len(data)
        want = oracle.encode_batch(oracle_tables["hpack"], 0xFF, data, offs, cap)
        total = int(want["out_offsets"][-1])
        for skew in (0, 5):  # the pinned buffer's first byte at two different 16-byte phases
            pinned = torch.zeros(cap + 64, dtype=torch.uint8).pin_memory().numpy()
            out = pinned[skew:skew + cap]
            got = ctx.encode(data, offs, cap, out=out)
            for k in ("out_offsets", "out_lens", "status", "consumed", "overflow_pattern", "overflow_num_bits"):
                assert np.array_equal(got[k], want[k]), k
            assert np.array_equal(out[:total], want["out"][:total])
            assert not pinned[:skew].any() and not pinned[skew + total:skew + total + 32].any()  # nothing outside
        stream = want["out"][:total]
        want_d = oracle.decode_batch(oracle_tables["hpack"], stream, want["out_offsets"], len(data) + 64)
        pinned = torch.zeros(len(data) + 128, dtype=torch.uint8).pin_memory().numpy()
        out = pinned[3:3 + len(data) + 64]
        got_d = ctx.decode(stream, want["out_offsets"], len(data) + 64, out=out)
        for k in ("out_offsets", "out_lens", "status", "consumed", "leftover_working_bits", "leftover_num_bits"):
            assert np.array_equal(got_d[k], want_d[k]), k
        assert np.array_equal(out[:len(data)], data)
        # too small by one byte: the call fails with SHORT_BUFFER, the offsets are complete
        small = torch.zeros(total - 1, dtype=torch.uint8).pin_memory().numpy()
        with pytest.raises(pkg.CodecError) as err:
            ctx.encode(data, offs, total - 1, out=small)
        assert err.value.code == pkg.AWS_ERROR_SHORT_BUFFER
        assert np.array_equal(err.value.result["out_offsets"], want["out_offsets"]) if hasattr(err.value, "result") else True
    finally:
        ctx.close()
