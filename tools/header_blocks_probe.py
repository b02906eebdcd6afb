#!/usr/bin/env python3
"""HPACK header blocks, device pointers: a seeded request mix of 256K header lists of 8-24 fields through
aws_hpack_header_block_encode_batch_device and _decode_batch_device, beside the string-literal calls on the same
names and values, so that the cost of the block layer is visible. One JSON line (profiles/r3_header_blocks.json).
With --records: the same lists through aws_hpack_header_block_encode_records_batch_device instead, with records from
an encoder-side dynamic table (EncoderTable of tests/hpack_records_oracle.py, 4096 octets) per connection of 64 consecutive lists, built on the
host and not timed; the blocks decode back to exactly those records (profiles/r3_header_block_records.json).

Mix per field: 25 % an exact Appendix A entry (indexed), 45 % an Appendix A name with a value, 30 % one of 32
custom names with a value; values of 8-256 octets of Zipf-sampled HPACK symbols (tests/refcodec.py); 5 % of the
fields never-indexed. The working set (about 0.4 GB of strings) is larger than the L2."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as graft  # noqa: E402
import hpack_records_oracle as _rec  # noqa: E402
import refcodec  # noqa: E402

_spec = importlib.util.spec_from_file_location(
    "hpack_header_block_oracle", os.path.join(ROOT, "oracle", "hpack_header_block_oracle.py"))
_blk = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(_blk)

CUSTOM_NAMES = [b"x-custom-header-%02d" % i for i in range(32)]


def synthetic_lists(n, seed, dev, static_table=None):
    """(field_offsets, strings, string_offsets, never_indexed) as device tensors (int64 offsets, uint8 data).
    static_table: the (name, value) entries of the exact and name matches (default: RFC 7541 Appendix A)."""
    static_table = _blk.STATIC_TABLE if static_table is None else static_table
    entries = len(static_table)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    counts = torch.randint(8, 25, (n,), generator=g, device=dev)
    fo = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    fo[1:] = torch.cumsum(counts, 0)
    F = int(fo[-1].item())
    # a pool of fixed strings: the static names and values, then the custom names
    pool, starts, lens = b"", [], []
    for s in [x for entry in static_table for x in entry] + CUSTOM_NAMES:
        starts.append(len(pool))
        lens.append(len(s))
        pool += s
    pool_t = torch.frombuffer(bytearray(pool), dtype=torch.uint8).to(dev)
    p_start = torch.tensor(starts, dtype=torch.int64, device=dev)
    p_len = torch.tensor(lens, dtype=torch.int64, device=dev)
    with_value = torch.tensor([i for i, (_, v) in enumerate(static_table) if v], dtype=torch.int64, device=dev)
    r = torch.rand(F, generator=g, device=dev)
    exact = r < 0.25
    custom = r >= 0.70
    entry = torch.where(exact, with_value[torch.randint(0, with_value.numel(), (F,), generator=g, device=dev)],
                        torch.randint(0, entries, (F,), generator=g, device=dev))
    name_id = torch.where(custom, 2 * entries + torch.randint(0, 32, (F,), generator=g, device=dev), 2 * entry)
    value_len = torch.where(exact, p_len[2 * entry + 1], torch.randint(8, 257, (F,), generator=g, device=dev))
    lens2 = torch.stack([p_len[name_id], value_len], 1).reshape(-1)
    so = torch.zeros(2 * F + 1, dtype=torch.int64, device=dev)
    so[1:] = torch.cumsum(lens2, 0)
    S = int(so[-1].item())
    # every output octet is a gather from [pool | random symbols]; random values read the random part at their own
    # output position
    sampler = torch.from_numpy(refcodec.zipf_symbol_sampler(refcodec.table_arrays("hpack")[1])).to(dev)
    rand = sampler[torch.randint(0, 65536, (S,), generator=g, device=dev)]
    src = torch.stack([p_start[name_id],
                       torch.where(exact, p_start[2 * entry + 1], pool_t.numel() + so[1:-1:2])], 1).reshape(-1)
    idx = torch.repeat_interleave(src - so[:-1], lens2) + torch.arange(S, device=dev)
    strings = torch.cat([pool_t, rand])[idx]
    del idx, rand
    never = (torch.rand(F, generator=g, device=dev) < 0.05).to(torch.uint8)
    return fo, strings, so, never


def round_trip(ctx, lists, dev, reps=1, stream=None):
    """Encode the lists into header blocks and decode them back; with reps > 1 also times both (CUDA events, first
    two repetitions are warm-up) and the string-literal calls on the same names and values."""
    fo, strings, so, never = lists
    n, F, S = fo.numel() - 1, (so.numel() - 1) // 2, strings.numel()
    stream = stream or torch.cuda.Stream(dev)
    out = torch.empty(S + 12 * F + 64, dtype=torch.uint8, device=dev)
    out_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    r = {"field_offsets": torch.zeros(n + 1, dtype=torch.int64, device=dev),
         "field_kind": torch.empty(F, dtype=torch.uint8, device=dev),
         "field_index": torch.empty(F, dtype=torch.int64, device=dev),
         "strings": torch.empty(S + 64, dtype=torch.uint8, device=dev),
         "string_offsets": torch.zeros(2 * F + 1, dtype=torch.int64, device=dev),
         "status": torch.ones(n, dtype=torch.int32, device=dev)}
    lit_framed = torch.empty(S + 20 * F + 64, dtype=torch.uint8, device=dev)
    lit_off = torch.zeros(2 * F + 1, dtype=torch.int64, device=dev)
    lit_out = torch.empty(S + 64, dtype=torch.uint8, device=dev)
    lit_out_off = torch.zeros(2 * F + 1, dtype=torch.int64, device=dev)
    lit_status = torch.zeros(2 * F, dtype=torch.int32, device=dev)
    times = {"encode": [], "decode": [], "lit_encode": [], "lit_decode": []}
    cs = stream.cuda_stream
    with torch.cuda.stream(stream):
        for rep in range(reps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record(stream)
            ctx.hpack_encode_blocks_device(n, fo, F, strings, so, S, out, out_off, mode=0, never_indexed=never, stream=cs)
            ev[1].record(stream)
            in_size = int(out_off[-1].item())
            ev2 = torch.cuda.Event(enable_timing=True)
            ev2.record(stream)
            ctx.hpack_decode_blocks_device(n, out, out_off, in_size, r["field_offsets"], r["field_kind"], r["field_index"],
                                           r["strings"], r["string_offsets"], status=r["status"], stream=cs)
            ev[2].record(stream)
            if reps > 1:
                lv = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
                lv[0].record(stream)
                ctx.hpack_device(True, 2 * F, strings, so, S, lit_framed, lit_framed.numel(), lit_off, mode=0, stream=cs)
                lv[1].record(stream)
                lit_size = int(lit_off[-1].item())
                lv[2].record(stream)
                ctx.hpack_device(False, 2 * F, lit_framed, lit_off, lit_size, lit_out, lit_out.numel(), lit_out_off,
                                 status=lit_status, stream=cs)
                lv[3].record(stream)
            torch.cuda.synchronize(dev)
            if rep >= 2:
                times["encode"].append(ev[0].elapsed_time(ev[1]))
                times["decode"].append(ev2.elapsed_time(ev[2]))
                times["lit_encode"].append(lv[0].elapsed_time(lv[1]))
                times["lit_decode"].append(lv[2].elapsed_time(lv[3]))
    if reps > 1:
        assert int(lit_status.abs().sum().item()) == 0 and torch.equal(lit_out[:S], strings)
    r.update(block_bytes=in_size, times=times)
    return r


def policy_records(lists, per_connection=64, max_size=4096):
    """Host arrays (field_offsets, field_kind, field_index, strings, string_offsets) of the records an encoder with its
    own dynamic table writes for the lists: a fresh EncoderTable every `per_connection` lists."""
    fo, strings, so, never = [t.cpu().numpy() for t in lists]
    fo, so, never, raw = fo.tolist(), so.tolist(), never.tolist(), strings.tobytes()
    blocks = []
    for b in range(len(fo) - 1):
        if b % per_connection == 0:
            table = _rec.EncoderTable(max_size)
        f0, f1 = fo[b], fo[b + 1]
        headers = [(raw[so[2 * f]:so[2 * f + 1]], raw[so[2 * f + 1]:so[2 * f + 2]]) for f in range(f0, f1)]
        blocks.append(table.records(headers, never[f0:f1]))
    return _rec.records_batch(blocks)


def records_leg(ctx, records, dev, reps=8, stream=None):
    """records through encode_records_batch_device (timed: CUDA events, first two repetitions are warm-up), then
    decoded back; returns the decoded arrays, the block size and the times."""
    fo, kind, index, strings, so = [torch.from_numpy(np.require(a, requirements="W").view(np.int64) if a.dtype == np.uint64
                                                     else np.require(a, requirements="W")).to(dev) for a in records]
    n, F, S = fo.numel() - 1, kind.numel(), strings.numel()
    stream = stream or torch.cuda.Stream(dev)
    out = torch.empty(S + 12 * F + 64, dtype=torch.uint8, device=dev)
    out_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    status = torch.ones(n, dtype=torch.int32, device=dev)
    r = {"field_offsets": torch.zeros(n + 1, dtype=torch.int64, device=dev),
         "field_kind": torch.empty(F, dtype=torch.uint8, device=dev),
         "field_index": torch.empty(F, dtype=torch.int64, device=dev),
         "strings": torch.empty(S + 64, dtype=torch.uint8, device=dev),
         "string_offsets": torch.zeros(2 * F + 1, dtype=torch.int64, device=dev),
         "status": torch.ones(n, dtype=torch.int32, device=dev)}
    times = []
    cs = stream.cuda_stream
    with torch.cuda.stream(stream):
        for rep in range(reps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record(stream)
            ctx.hpack_encode_records_device(n, fo, F, kind, index, strings, so, S, out, out_off, status, mode=0,
                                            stream=cs)
            ev[1].record(stream)
            torch.cuda.synchronize(dev)
            if rep >= 2:
                times.append(ev[0].elapsed_time(ev[1]))
        in_size = int(out_off[-1].item())
        ctx.hpack_decode_blocks_device(n, out, out_off, in_size, r["field_offsets"], r["field_kind"], r["field_index"],
                                       r["strings"], r["string_offsets"], status=r["status"], stream=cs)
        torch.cuda.synchronize(dev)
    assert int(status.abs().sum().item()) == 0 and int(r["status"].abs().sum().item()) == 0
    assert torch.equal(r["field_offsets"], fo) and torch.equal(r["field_kind"], kind)
    assert torch.equal(r["field_index"], index) and torch.equal(r["string_offsets"], so)
    assert torch.equal(r["strings"][:S], strings)
    return {"block_bytes": in_size, "times": times, "fields": F}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                        text=True, timeout=60).strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    records_mode = "--records" in sys.argv
    pkg = graft.load_package()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n = 262_144
    lists = synthetic_lists(n, 1, dev)
    fo, strings, so, never = lists
    F, S = (so.numel() - 1) // 2, strings.numel()
    ctx = pkg.BatchContext(pkg.coders_library().coder("hpack"), eos_padding=0xFF, device=0)
    if records_mode:
        records = policy_records(lists)
    r = round_trip(ctx, lists, dev, reps=8)
    assert int(r["status"].abs().sum().item()) == 0 and torch.equal(r["field_offsets"], fo)
    assert torch.equal(r["string_offsets"], so) and torch.equal(r["strings"][:S], strings)
    t = {k: float(np.median(v)) for k, v in r["times"].items()}
    moved = r["block_bytes"] + S
    name, power = card()
    if records_mode:
        k = records_leg(ctx, records, dev)
        kinds = np.bincount(records[1], minlength=5)
        print(json.dumps({
            "workload": "hpack header blocks from records (RFC 7541 2.3, 4, 6): the lists of r3_header_blocks.json, "
                        "records of an encoder-side dynamic table of 4096 octets per connection of 64 lists (built on "
                        "the host, not timed), SMALLEST mode, device pointers",
            "header_lists": n, "connections": (n + 63) // 64, "fields": F, "string_bytes": S,
            "records": {"indexed_static": int(((records[1] == 0) & (records[2] <= 61)).sum()),
                        "indexed_dynamic": int(((records[1] == 0) & (records[2] > 61)).sum()),
                        "incremental": int(kinds[1]), "never_indexed": int(kinds[3])},
            "block_bytes": k["block_bytes"], "stateless_block_bytes": r["block_bytes"],
            "encode_records_ms": float(np.median(k["times"])), "stateless_encode_ms": t["encode"],
            "round_trip": "decoded records identical to the encoded ones",
            "repetitions": len(k["times"]), "statistic": "median after 2 warm-up repetitions",
            "gpu": name, "power_limit": power}))
        ctx.close()
        return
    print(json.dumps({
        "workload": "hpack header blocks (RFC 7541 6), %d header lists of 8-24 fields (25%% exact static, 45%% static "
                    "name, 30%% custom name; values 8-256 B Zipf), SMALLEST mode, device pointers" % n,
        "fields": F, "string_bytes": S, "block_bytes": r["block_bytes"],
        "encode_ms": t["encode"], "decode_ms": t["decode"],
        "encode_gbs": moved / t["encode"] / 1e6, "decode_gbs": moved / t["decode"] / 1e6,
        "literals_encode_ms": t["lit_encode"], "literals_decode_ms": t["lit_decode"],
        "literals_note": "aws_hpack_string_*_batch_device on all %d names and values of the same lists" % (2 * F),
        "repetitions": len(r["times"]["encode"]), "statistic": "median after 2 warm-up repetitions",
        "gpu": name, "power_limit": power}))
    ctx.close()


if __name__ == "__main__":
    main()
