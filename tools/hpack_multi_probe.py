#!/usr/bin/env python3
"""HPACK literals and header blocks over several GPUs, host pointers: the five _multi calls on the 256K header lists
of tools/header_blocks_probe.py (synthetic_lists: 4.2M fields), on 1, 2, 4 and 8 contexts, one per GPU (capped at the
GPUs present). One JSON line (profiles/r4_hpack_multi.json).

Before any timing, every call over all contexts is checked array for array against the single-context call. Each call
is timed end to end with a host clock (the calls synchronise): median of 6 runs after 2 warm-ups. Beside each, the same
number of GPUs runs the copies alone: the call's input octets host to device and its output octets device to host,
split over the GPUs as the call's shards split them, no kernels (the copies_alone baseline of DESIGN.md section 6).
Inputs of the calls other than block encode are the single-context outputs: blocks and literals from the encoders,
records from the block decoder."""
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import header_blocks_probe as hbp  # noqa: E402

graft = hbp.graft
WARMUP, RUNS = 2, 6


def _p(a):
    return a.ctypes.data


class Probe:
    def __init__(self, pkg, lists):
        self.capi = pkg.capi
        self.fo, self.strings, self.so, self.never = lists
        self.n, self.F, self.S = len(self.fo) - 1, len(self.never), len(self.strings)

    def _run(self, target, name, *args):
        err = self.capi.hpack_host_call(target, name, *args)
        if err:
            raise RuntimeError("%s: aws error %d" % (name, err))

    def block_encode(self, target):
        out, off = np.empty(self.S + 32 * self.F + 64, np.uint8), np.empty(self.n + 1, np.uint64)
        lists = self.capi.aws_hpack_header_lists(self.n, _p(self.fo), 0, None, None, _p(self.never), _p(self.strings), 0,
                                                 _p(self.so))
        self._run(target, "aws_hpack_header_block_encode_batch", C.byref(lists), 0, _p(out), len(out), _p(off))
        return {"out": out[:int(off[-1])], "out_offsets": off}

    def block_decode(self, target, blocks, offs):
        r = {"field_offsets": np.empty(self.n + 1, np.uint64), "field_kind": np.empty(self.F, np.uint8),
             "field_index": np.empty(self.F, np.uint64), "strings": np.empty(self.S + 64, np.uint8),
             "string_offsets": np.empty(2 * self.F + 1, np.uint64), "status": np.empty(self.n, np.int32)}
        lists = self.capi.aws_hpack_header_lists(self.n, _p(r["field_offsets"]), self.F, _p(r["field_kind"]),
                                                 _p(r["field_index"]), None, _p(r["strings"]), len(r["strings"]),
                                                 _p(r["string_offsets"]))
        self._run(target, "aws_hpack_header_block_decode_batch", self.n, _p(blocks), _p(offs), C.byref(lists),
                  _p(r["status"]))
        r["strings"] = r["strings"][:self.S]
        return r

    def records_encode(self, target, kind, index):
        out, off, st = np.empty(self.S + 32 * self.F + 64, np.uint8), np.empty(self.n + 1, np.uint64), np.empty(self.n, np.int32)
        lists = self.capi.aws_hpack_header_lists(self.n, _p(self.fo), 0, _p(kind), _p(index), _p(self.never),
                                                 _p(self.strings), 0, _p(self.so))
        self._run(target, "aws_hpack_header_block_encode_records_batch", C.byref(lists), 0, _p(out), len(out), _p(off),
                  _p(st))
        return {"out": out[:int(off[-1])], "out_offsets": off, "status": st}

    def string_encode(self, target):
        out, off = np.empty(self.S + 20 * self.F + 64, np.uint8), np.empty(2 * self.F + 1, np.uint64)
        self._run(target, "aws_hpack_string_encode_batch", 2 * self.F, _p(self.strings), _p(self.so), 0, _p(out), len(out),
                  _p(off))
        return {"out": out[:int(off[-1])], "out_offsets": off}

    def string_decode(self, target, framed, offs):
        out, off, st = np.empty(self.S + 64, np.uint8), np.empty(2 * self.F + 1, np.uint64), np.empty(2 * self.F, np.int32)
        self._run(target, "aws_hpack_string_decode_batch", 2 * self.F, _p(framed), _p(offs), _p(out), len(out), _p(off),
                  _p(st))
        return {"out": out[:int(off[-1])], "out_offsets": off, "status": st}


def timed(fn):
    times = []
    for rep in range(WARMUP + RUNS):
        t0 = time.perf_counter()
        fn()
        if rep >= WARMUP:
            times.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(times)


def copies_alone(gpus, in_bytes, out_bytes, weight, library):
    """Median ms of the copies alone: in_bytes host to device and out_bytes back, split over `gpus` GPUs by the shard
    plan of `weight`, one host thread per GPU, pageable host memory as the caller's."""
    begin = library.plan_shards(weight, gpus)
    share = [(int(weight[begin[d + 1]]) - int(weight[begin[d]])) / max(1, int(weight[-1])) for d in range(gpus)]
    ins = [int(in_bytes * s) for s in share]
    outs = [int(out_bytes * s) for s in share]
    host_in, host_out = np.ones(sum(ins), np.uint8), np.ones(sum(outs), np.uint8)
    at_in, at_out = np.cumsum([0] + ins), np.cumsum([0] + outs)
    dev = [(torch.empty(ins[d], dtype=torch.uint8, device=d), torch.empty(outs[d], dtype=torch.uint8, device=d))
           for d in range(gpus)]

    def one(d):
        torch.cuda.set_device(d)
        dev[d][0].copy_(torch.from_numpy(host_in[at_in[d]:at_in[d + 1]]))
        torch.from_numpy(host_out[at_out[d]:at_out[d + 1]]).copy_(dev[d][1])
        torch.cuda.synchronize(d)

    def run():
        threads = [threading.Thread(target=one, args=(d,)) for d in range(gpus)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
    return timed(run)


def same(a, b, what):
    for key in a:
        if not np.array_equal(a[key], b[key]):
            raise AssertionError("%s: %s differs from the single-context call" % (what, key))


def main():
    pkg = graft.load_package()
    available = torch.cuda.device_count()
    counts = [k for k in (1, 2, 4, 8) if k <= available]
    n = 262_144
    lists = [t.cpu().numpy() for t in hbp.synthetic_lists(n, 1, torch.device("cuda", 0))]
    lists = [a.view(np.uint64) if a.dtype == np.int64 else a for a in lists]
    ctxs = [pkg.BatchContext(pkg.coders_library().coder("hpack"), eos_padding=0xFF, device=d) for d in range(max(counts))]
    # (parity over two contexts at least: a second one on device 0 when the box has one GPU)
    pair = ctxs if len(ctxs) > 1 else ctxs + [pkg.BatchContext(pkg.coders_library().coder("hpack"), 0xFF, device=0)]
    p = Probe(pkg, lists)
    one = ctxs[0]
    # inputs from the single-context calls
    enc = p.block_encode(one)
    dec = p.block_decode(one, enc["out"], enc["out_offsets"])
    assert not dec["status"].any() and np.array_equal(dec["field_offsets"], p.fo) and np.array_equal(dec["strings"], p.strings)
    kind, index = dec["field_kind"], dec["field_index"]
    rec = p.records_encode(one, kind, index)
    lit = p.string_encode(one)
    lit_dec = p.string_decode(one, lit["out"], lit["out_offsets"])
    assert not lit_dec["status"].any() and np.array_equal(lit_dec["out"], p.strings)
    # the five calls: (run on a target, the single-context result, input octets, output octets, shard weights)
    list_octets = p.so[2 * p.fo]
    blocks_in, lits_in = len(enc["out"]) + 8 * (n + 1), len(lit["out"]) + 8 * (2 * p.F + 1)
    fields_in = 8 * (n + 1) + p.S + 8 * (2 * p.F + 1) + p.F
    fields_out = 8 * (n + 1) + 4 * n + 9 * p.F + p.S + 8 * (2 * p.F + 1)
    calls = {
        "block_encode": (lambda t: p.block_encode(t), enc, fields_in, len(enc["out"]) + 8 * (n + 1), list_octets),
        "block_encode_records": (lambda t: p.records_encode(t, kind, index), rec, fields_in + 9 * p.F,
                                 len(rec["out"]) + 8 * (n + 1) + 4 * n, list_octets),
        "block_decode": (lambda t: p.block_decode(t, enc["out"], enc["out_offsets"]), dec, blocks_in, fields_out,
                         enc["out_offsets"]),
        "string_encode": (lambda t: p.string_encode(t), lit, 8 * (2 * p.F + 1) + p.S, lits_in, p.so),
        "string_decode": (lambda t: p.string_decode(t, lit["out"], lit["out_offsets"]), lit_dec, lits_in,
                          p.S + 8 * (2 * p.F + 1) + 8 * p.F, lit["out_offsets"]),
    }
    for name, (run, want, _, _, _) in calls.items():
        same(run(pair), want, name)  # over every context, before any timing
    result = {}
    for name, (run, _, in_bytes, out_bytes, weight) in calls.items():
        rows = []
        for k in counts:
            ms = timed(lambda: run(ctxs[:k]))
            base = copies_alone(k, in_bytes, out_bytes, weight, ctxs[0].library)
            rows.append({"gpus": k, "call_ms": ms, "copies_alone_ms": base})
        for row in rows:
            row["speedup_vs_1_gpu"] = rows[0]["call_ms"] / row["call_ms"]
            row["copies_alone_speedup_vs_1_gpu"] = rows[0]["copies_alone_ms"] / row["copies_alone_ms"]
            row["call_over_copies_alone"] = row["call_ms"] / row["copies_alone_ms"]
        result[name] = {"input_bytes": int(in_bytes), "output_bytes": int(out_bytes), "by_gpus": rows}
    gpu, power = hbp.card()
    print(json.dumps({
        "workload": "the %d header lists of r3_header_blocks.json (%d fields, %d string octets), SMALLEST mode, host "
                    "pointers, one context per GPU; string calls on all %d names and values" % (n, p.F, p.S, 2 * p.F),
        "parity": "every call over %d contexts identical to the single-context call, array for array" % len(pair),
        "calls": result, "statistic": "median of %d end-to-end host-clock runs after %d warm-ups" % (RUNS, WARMUP),
        "gpu": gpu, "power_limit": power, "gpu_count": available}))
    for c in set(pair):
        c.close()


if __name__ == "__main__":
    main()
