#!/usr/bin/env python3
"""QPACK field sections, device pointers: the request mix of tools/header_blocks_probe.py (256K header lists of 8-24
fields; 25 % exact static entries, 45 % static names with a value, 30 % custom names; values of 8-256 octets of
Zipf-sampled HPACK symbols; 5 % never-indexed), with RFC 9204 Appendix A as the static table, through
aws_qpack_field_section_encode_batch_device and _decode_batch_device, beside the string-literal calls on the same names
and values, so that the cost of the section layer is visible. The decoded lists are checked against the encoded ones
before anything is printed. One JSON line (profiles/r5_qpack_sections.json)."""
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
_q = _load("qpack_field_section_oracle", "oracle", "qpack_field_section_oracle.py")


def synthetic_lists(n, seed, dev):
    """(field_offsets, strings, string_offsets, never_indexed) as device tensors (int64 offsets, uint8 data)."""
    return _hb.synthetic_lists(n, seed, dev, static_table=_q.STATIC_TABLE)


def round_trip(ctx, lists, dev, reps=1, stream=None):
    """Encode the lists into field sections and decode them back; with reps > 1 also times both (CUDA events, first
    two repetitions are warm-up) and the string-literal calls on the same names and values."""
    fo, strings, so, never = lists
    n, F, S = fo.numel() - 1, (so.numel() - 1) // 2, strings.numel()
    stream = stream or torch.cuda.Stream(dev)
    out = torch.empty(S + 12 * F + 2 * n + 64, dtype=torch.uint8, device=dev)
    out_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    r = {"encoded_insert_count": torch.ones(n, dtype=torch.int64, device=dev),
         "base_sign": torch.ones(n, dtype=torch.uint8, device=dev),
         "delta_base": torch.ones(n, dtype=torch.int64, device=dev),
         "field_offsets": torch.zeros(n + 1, dtype=torch.int64, device=dev),
         "field_kind": torch.empty(F, dtype=torch.uint8, device=dev),
         "field_index": torch.empty(F, dtype=torch.int64, device=dev),
         "never_indexed": torch.empty(F, dtype=torch.uint8, device=dev),
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
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            ev[0].record(stream)
            ctx.qpack_encode_sections_device(n, fo, F, strings, so, S, out, out_off, mode=0, never_indexed=never,
                                             stream=cs)
            ev[1].record(stream)
            in_size = int(out_off[-1].item())
            ev[2].record(stream)
            ctx.qpack_decode_sections_device(n, out, out_off, in_size, r["encoded_insert_count"], r["base_sign"],
                                             r["delta_base"], r["field_offsets"], r["field_kind"], r["field_index"],
                                             r["never_indexed"], r["strings"], r["string_offsets"], status=r["status"],
                                             stream=cs)
            ev[3].record(stream)
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
                times["decode"].append(ev[2].elapsed_time(ev[3]))
                times["lit_encode"].append(lv[0].elapsed_time(lv[1]))
                times["lit_decode"].append(lv[2].elapsed_time(lv[3]))
    if reps > 1:
        assert int(lit_status.abs().sum().item()) == 0 and torch.equal(lit_out[:S], strings)
    r.update(section_bytes=in_size, times=times)
    return r


def main():
    pkg = graft.load_package()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n = 262_144
    lists = synthetic_lists(n, 1, dev)
    fo, strings, so, never = lists
    F, S = (so.numel() - 1) // 2, strings.numel()
    ctx = pkg.BatchContext(pkg.coders_library().coder("hpack"), eos_padding=0xFF, device=0)
    r = round_trip(ctx, lists, dev, reps=8)
    # the round trip: every section decodes without error to the lists that were encoded
    assert int(r["status"].abs().sum().item()) == 0 and torch.equal(r["field_offsets"], fo)
    assert torch.equal(r["string_offsets"], so) and torch.equal(r["strings"][:S], strings)
    assert torch.equal(r["never_indexed"], never)
    assert int(r["encoded_insert_count"].abs().sum().item()) == 0 and int(r["delta_base"].abs().sum().item()) == 0
    kinds = torch.bincount(r["field_kind"].to(torch.int64), minlength=7).tolist()
    t = {k: float(np.median(v)) for k, v in r["times"].items()}
    moved = r["section_bytes"] + S
    name, power = _hb.card()
    print(json.dumps({
        "workload": "qpack field sections (RFC 9204 4.5), %d header lists of 8-24 fields (25%% exact static, 45%% "
                    "static name, 30%% custom name; values 8-256 B Zipf), SMALLEST mode, device pointers" % n,
        "fields": F, "string_bytes": S, "section_bytes": r["section_bytes"],
        "lines": {"indexed_static": kinds[0], "name_ref_static": kinds[3], "literal_name": kinds[6]},
        "encode_ms": t["encode"], "decode_ms": t["decode"],
        "encode_gbs": moved / t["encode"] / 1e6, "decode_gbs": moved / t["decode"] / 1e6,
        "literals_encode_ms": t["lit_encode"], "literals_decode_ms": t["lit_decode"],
        "literals_note": "aws_hpack_string_*_batch_device on all %d names and values of the same lists" % (2 * F),
        "round_trip": "decoded lists identical to the encoded ones",
        "repetitions": len(r["times"]["encode"]), "statistic": "median after 2 warm-up repetitions",
        "gpu": name, "power_limit": power}))
    ctx.close()


if __name__ == "__main__":
    main()
