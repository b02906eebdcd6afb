#!/usr/bin/env python3
"""QPACK encoder- and decoder-stream instructions, device pointers. Encoder stream: 256K chunks (one per connection)
built from the header lists of tools/qpack_sections_probe.py (8-24 instructions each, about 4M in all): the first
instruction of every chunk is a Set Dynamic Table Capacity, 5 % of the others are Duplicates, and the rest are
INSERT_AUTO on the lists' names and values (so 25 % + 45 % of them become static name references and 30 % literal
names, values of 8-256 octets of Zipf-sampled HPACK symbols). Decoder stream: one chunk per connection of 1-4 Section
Acknowledgments, Stream Cancellations and Insert Count Increments. Both go through
aws_qpack_instruction_encode_batch_device and _decode_batch_device, the encoder stream beside the string-literal
calls on the same names and values, so that the cost of the instruction layer is visible. The decoded records are
checked against the encoded ones before anything is printed. One JSON line (profiles/r6_qpack_instructions.json);
--profile prints the per-kernel split of one round trip from torch.profiler instead
(profiles/r6_qpack_instructions_kernels.json)."""
import importlib.util
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as graft  # noqa: E402


def _load(name, *path):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, *path))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module


_hb = _load("header_blocks_probe", "tools", "header_blocks_probe.py")
_qs = _load("qpack_sections_probe", "tools", "qpack_sections_probe.py")
ENC, DEC = 0, 1
IS, ID, IL, DUP, CAP, ACK, CANCEL, ICI, AUTO = range(9)


def _drop_strings(strings, so, keep):
    """The packed strings with those of the instructions where keep is False emptied: (strings, string_offsets)."""
    lens = (so[1:] - so[:-1]) * keep.repeat_interleave(2).to(torch.int64)
    new_so = torch.zeros_like(so)
    new_so[1:] = torch.cumsum(lens, 0)
    seg = torch.repeat_interleave(torch.arange(lens.numel(), device=so.device), lens)
    src = so[seg] + (torch.arange(seg.numel(), device=so.device) - new_so[seg])
    return strings[src], new_so


def synthetic_streams(n, seed, dev):
    """((instruction_offsets, kind, index, strings, string_offsets) of the encoder stream, the same of the decoder
    stream) as device tensors (int64 offsets and indices, uint8 kinds and data)."""
    fo, strings, so, _ = _qs.synthetic_lists(n, seed, dev)
    F = int(fo[-1].item())
    g = torch.Generator(device=dev)
    g.manual_seed(seed + 1)
    kind = torch.full((F,), AUTO, dtype=torch.uint8, device=dev)
    index = torch.zeros(F, dtype=torch.int64, device=dev)
    dup = torch.rand(F, generator=g, device=dev) < 0.05
    kind[dup] = DUP
    index[dup] = torch.randint(0, 20, (F,), generator=g, device=dev)[dup]
    first = fo[:-1]
    kind[first] = CAP
    index[first] = torch.randint(0, 65536, (n,), generator=g, device=dev)
    strings, so = _drop_strings(strings, so, kind == AUTO)
    counts = torch.randint(1, 5, (n,), generator=g, device=dev)
    dfo = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    dfo[1:] = torch.cumsum(counts, 0)
    D = int(dfo[-1].item())
    dkind = (ACK + torch.randint(0, 3, (D,), generator=g, device=dev)).to(torch.uint8)
    dindex = 4 * torch.randint(0, 1 << 20, (D,), generator=g, device=dev)
    dindex = torch.where(dkind == ICI, 1 + torch.randint(0, 200, (D,), generator=g, device=dev), dindex)
    dso = torch.zeros(2 * D + 1, dtype=torch.int64, device=dev)
    return (fo, kind, index, strings, so), (dfo, dkind, dindex, torch.zeros(0, dtype=torch.uint8, device=dev), dso)


def round_trip(ctx, which, batch, dev, reps=1, stream=None, literals=False):
    """Encode the instructions into chunks of the stream `which` and decode them back; with reps > 1 also times both
    (CUDA events, the first two repetitions are warm-up) and, with literals, the string-literal calls on the same
    names and values."""
    io_, kind, index, strings, so = batch
    n, F, S = io_.numel() - 1, (so.numel() - 1) // 2, strings.numel()
    stream = stream or torch.cuda.Stream(dev)
    out = torch.empty(S + 12 * F + 64, dtype=torch.uint8, device=dev)
    r = {"out_offsets": torch.zeros(n + 1, dtype=torch.int64, device=dev),
         "instruction_offsets": torch.zeros(n + 1, dtype=torch.int64, device=dev),
         "kind": torch.empty(F, dtype=torch.uint8, device=dev), "index": torch.empty(F, dtype=torch.int64, device=dev),
         "strings": torch.empty(S + 64, dtype=torch.uint8, device=dev),
         "string_offsets": torch.zeros(2 * F + 1, dtype=torch.int64, device=dev),
         "consumed": torch.ones(n, dtype=torch.int64, device=dev), "status": torch.ones(n, dtype=torch.int32, device=dev),
         "enc_status": torch.ones(n, dtype=torch.int32, device=dev)}
    if literals:
        lit_framed = torch.empty(S + 20 * F + 64, dtype=torch.uint8, device=dev)
        lit_off = torch.zeros(2 * F + 1, dtype=torch.int64, device=dev)
        lit_out = torch.empty(S + 64, dtype=torch.uint8, device=dev)
        lit_out_off = torch.zeros(2 * F + 1, dtype=torch.int64, device=dev)
        lit_status = torch.zeros(2 * F, dtype=torch.int32, device=dev)
    times = {"encode": [], "decode": [], "lit_encode": [], "lit_decode": []}
    cs = stream.cuda_stream
    with torch.cuda.stream(stream):
        for rep in range(reps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            ev[0].record(stream)
            ctx.qpack_encode_instructions_device(which, n, io_, F, kind, index, strings, so, S, out, r["out_offsets"],
                                                 status=r["enc_status"], mode=0, stream=cs)
            ev[1].record(stream)
            in_size = int(r["out_offsets"][-1].item())
            ev[2].record(stream)
            ctx.qpack_decode_instructions_device(which, n, out, r["out_offsets"], in_size, r["instruction_offsets"],
                                                 r["kind"], r["index"], r["strings"], r["string_offsets"], r["consumed"],
                                                 status=r["status"], stream=cs)
            ev[3].record(stream)
            if literals:
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
                times["decode"].append(ev[2].elapsed_time(ev[3]))
                if literals:
                    times["lit_encode"].append(lv[0].elapsed_time(lv[1]))
                    times["lit_decode"].append(lv[2].elapsed_time(lv[3]))
    if literals:
        assert int(lit_status.abs().sum().item()) == 0 and torch.equal(lit_out[:S], strings)
    assert int(r["enc_status"].abs().sum().item()) == 0
    r.update(stream_bytes=in_size, times=times)
    return r


def _check(r, batch):
    io_, kind, index, strings, so = batch
    F = int(io_[-1].item())
    assert int(r["status"].abs().sum().item()) == 0
    assert torch.equal(r["consumed"], r["out_offsets"][1:] - r["out_offsets"][:-1])
    assert torch.equal(r["instruction_offsets"], io_) and torch.equal(r["string_offsets"], so)
    assert torch.equal(r["strings"][:strings.numel()], strings)
    explicit = kind != AUTO
    assert torch.equal(r["kind"][explicit], kind[explicit]) and torch.equal(r["index"][explicit], index[explicit])
    return torch.bincount(r["kind"][:F].to(torch.int64), minlength=8).tolist()


def profile(ctx, streams, dev):
    """Per-kernel device time of one round trip of each stream (after two unprofiled ones), from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile as torch_profile
    for which, batch in zip((ENC, DEC), streams):
        round_trip(ctx, which, batch, dev, reps=2)
    with torch_profile(activities=[ProfilerActivity.CUDA]) as prof:
        for which, batch in zip((ENC, DEC), streams):
            round_trip(ctx, which, batch, dev)
        torch.cuda.synchronize(dev)
    kernels = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            kernels[e.key] = {"ms": t / 1000.0, "calls": e.count}
    return dict(sorted(kernels.items(), key=lambda kv: -kv[1]["ms"]))


def main():
    pkg = graft.load_package()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n = 262_144
    streams = synthetic_streams(n, 1, dev)
    ctx = pkg.BatchContext(pkg.coders_library().coder("hpack"), eos_padding=0xFF, device=0)
    name, power = _hb.card()
    if "--profile" in sys.argv:
        print(json.dumps({"workload": "one round trip of each stream of tools/qpack_instructions_probe.py",
                          "kernels": profile(ctx, streams, dev), "source": "torch.profiler, CUDA activities",
                          "gpu": name, "power_limit": power}))
        ctx.close()
        return
    enc = round_trip(ctx, ENC, streams[0], dev, reps=8, literals=True)
    enc_kinds = _check(enc, streams[0])
    dec = round_trip(ctx, DEC, streams[1], dev, reps=8)
    dec_kinds = _check(dec, streams[1])
    t = {k: float(np.median(v)) for k, v in enc["times"].items() if v}
    td = {k: float(np.median(v)) for k, v in dec["times"].items() if v}
    io_, _, _, strings, so = streams[0]
    F, S = int(io_[-1].item()), strings.numel()
    moved = enc["stream_bytes"] + S
    print(json.dumps({
        "workload": "qpack encoder stream (RFC 9204 4.3), %d chunks of 8-24 instructions: a Set Dynamic Table "
                    "Capacity first, 5%% Duplicates, the rest INSERT_AUTO on the lists of tools/qpack_sections_probe.py "
                    "(25%% exact static, 45%% static name, 30%% custom name; values 8-256 B Zipf); decoder stream "
                    "(4.4), one chunk of 1-4 acknowledgments, cancellations and increments per connection; SMALLEST "
                    "mode, device pointers" % n,
        "encoder_instructions": F, "string_bytes": S, "encoder_stream_bytes": enc["stream_bytes"],
        "encoder_kinds": {"insert_name_ref_static": enc_kinds[IS], "insert_literal_name": enc_kinds[IL],
                          "duplicate": enc_kinds[DUP], "set_capacity": enc_kinds[CAP]},
        "encode_ms": t["encode"], "decode_ms": t["decode"],
        "encode_gbs": moved / t["encode"] / 1e6, "decode_gbs": moved / t["decode"] / 1e6,
        "literals_encode_ms": t["lit_encode"], "literals_decode_ms": t["lit_decode"],
        "literals_note": "aws_hpack_string_*_batch_device on all %d names and values of the encoder stream "
                         "(empty ones included)" % (2 * F),
        "decoder_instructions": int(streams[1][0][-1].item()), "decoder_stream_bytes": dec["stream_bytes"],
        "decoder_kinds": {"section_acknowledgment": dec_kinds[ACK], "stream_cancellation": dec_kinds[CANCEL],
                          "insert_count_increment": dec_kinds[ICI]},
        "decoder_encode_ms": td["encode"], "decoder_decode_ms": td["decode"],
        "round_trip": "decoded records identical to the encoded ones, consumed == chunk sizes",
        "repetitions": len(enc["times"]["encode"]), "statistic": "median after 2 warm-up repetitions",
        "gpu": name, "power_limit": power}))
    ctx.close()


if __name__ == "__main__":
    main()
