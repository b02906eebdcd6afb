"""The device-pointer entry points at caller-chosen addresses, exact capacities and on caller streams.

The host-pointer calls stage every array through buffers the context owns: 16-byte aligned, with slack after the
output and leftovers of earlier calls around the input. So they cannot show what the `_device` calls promise a
caller: any byte phase for `in` and `out` (several routes turn on `in & 15` and `out & 15`), no write past
`out + out_capacity` or past entry n of a per-item array, and results that do not depend on the bytes next to an item.

Every caller array here lives in its own device allocation behind and before a guard of seeded canary bytes (never
0x00 or 0xFF, so a stray write of either shows). After each call, on the caller's stream, every guard is
byte-identical to its canary and every input array is unchanged. The bytes directly around an input payload are
chosen by the test (0x00, 0xFF, or the payload's own first and last 16 bytes) and the result must not depend on
them. Each Huffman case also asserts, by the context's launch count, which route it ran. Everything is compared bit
for bit with the oracle (tests/refcodec.py and oracle/hpack_literals_oracle.py)."""
import itertools

import numpy as np
import pytest

import refcodec
from refcodec import OK, SHORT_BUFFER
from test_gpu_code_tables import batch, damaged, flip_bits, offsets, slots_around, table_arrays, with_runs
from test_hpack_literals import _strings, lit, literal_oracle  # noqa: F401 (literal_oracle is a fixture)

pytestmark = pytest.mark.gpu

GUARD = 64  # canary bytes before (plus the phase) and after every array
P64, P32, P8 = 8, 4, 3  # phases of 64-bit, 32-bit and byte per-item arrays: naturally aligned, not 16-byte aligned
FILLS = ("zero", "ones", "echo")
ALIGNED_IN = [(0, 0), (0, 1), (0, 5), (0, 15)]  # (in phase, out phase)
SHIFTED_IN = [(1, 0), (3, 3), (8, 1), (15, 15)]
CAPACITIES = ("need", "need-1", "half", "generous")
SWITCHES = ("AWS_HUFFMAN_BATCH_FORCE_GENERIC", "AWS_HUFFMAN_BATCH_NO_FUSED_STREAM", "AWS_HUFFMAN_BATCH_NO_STRINGS",
            "AWS_HUFFMAN_BATCH_NO_SLOTS")

_CANARY = np.random.default_rng(0xCA7A).integers(1, 255, size=1 << 16, dtype=np.uint8)
_placed = itertools.count()


def canary(size):
    """Seeded bytes in 1..254, a different stretch for every array."""
    return np.resize(np.roll(_CANARY, -(next(_placed) * 7919 % len(_CANARY))), size)


class Placed:
    """One caller array in its own device allocation: a front guard, `phase` bytes, the array, a back guard. For an
    input payload, `fill` sets the 16 bytes directly before and after it (inside the guards)."""

    def __init__(self, array, phase, fill=None):
        import torch
        array = np.ascontiguousarray(array)
        self.dtype = array.dtype
        raw = array.view(np.uint8).ravel()
        self.start = GUARD + phase
        self.end = self.start + raw.size
        self.image = canary(self.end + GUARD)
        self.image[self.start:self.end] = raw
        if fill is not None and raw.size:
            before = {"zero": np.zeros(16, np.uint8), "ones": np.full(16, 0xFF, np.uint8), "echo": raw[-16:]}[fill]
            after = {"zero": before, "ones": before, "echo": raw[:16]}[fill]
            self.image[self.start - len(before):self.start] = before
            self.image[self.end:self.end + len(after)] = after
        self.buf = torch.from_numpy(self.image.copy()).to("cuda:0")

    def data_ptr(self):
        return self.buf.data_ptr() + self.start

    def read(self, what, unchanged=False):
        """The array as the device holds it now; asserts that both guards (and, for an input, the array) are as
        placed."""
        got = self.buf.cpu().numpy()
        for name, a, b in (("front guard", 0, self.start), ("back guard", self.end, len(got))):
            bad = np.flatnonzero(got[a:b] != self.image[a:b])
            assert not len(bad), "%s: %s written at %s" % (what, name, (bad[:8] + a - self.start).tolist())
        if unchanged:
            bad = np.flatnonzero(got[self.start:self.end] != self.image[self.start:self.end])
            assert not len(bad), "%s: input changed at byte %s" % (what, bad[:8].tolist())
        return got[self.start:self.end].view(self.dtype)


def place(array, phase, fill=None):
    return Placed(array, phase, fill)


def scratch_array(dtype, count, phase):
    """An output array whose every entry starts as canary bytes (so an entry the call does not write shows)."""
    return Placed(canary(count * np.dtype(dtype).itemsize).view(dtype), phase)


def capacity(kind, need):
    return {"need": need, "need-1": need - 1, "half": need // 2, "generous": need + 4096}[kind]


def launches(ctx, call):
    before = ctx.launch_count
    call()
    return ctx.launch_count - before


# ---------------------------------------------------------------------------------------------------------------
# fixtures
# ---------------------------------------------------------------------------------------------------------------

@pytest.fixture
def stream(pkg):
    """A non-default stream, current for the whole test: placements, calls and read-backs are ordered on it."""
    import torch
    st = torch.cuda.Stream(torch.device("cuda", 0))
    with torch.cuda.stream(st):
        yield st
    st.synchronize()


@pytest.fixture(scope="module")
def tables(oracle, ref_free_masked_coder):
    made = {}

    def get(name):
        if name not in made:
            if name == "masked":
                arrays = ref_free_masked_coder[1:]
            elif name in ("hpack", "test"):
                arrays = refcodec.table_arrays(name)
            else:
                arrays = table_arrays(name)
            made[name] = oracle.table(*arrays)
        return made[name]
    return get


@pytest.fixture(scope="module")
def contexts(pkg, coders, ref_free_masked_coder):
    """contexts(table, eos, switch): hpack / test from the generated coders, masked from the Python callback coder,
    any other name from test_gpu_code_tables' code table; `switch` set (and no other) while the context is made."""
    made = {}

    def get(name, eos=0xFF, switch=None):
        key = (name, eos, switch)
        if key not in made:
            with pytest.MonkeyPatch.context() as mp:
                for var in SWITCHES:
                    mp.delenv(var, raising=False)
                if switch:
                    mp.setenv(switch, "1")
                if name in ("hpack", "test"):
                    made[key] = pkg.BatchContext(coders.coder(name), eos_padding=eos, device=0)
                elif name == "masked":
                    made[key] = pkg.BatchContext(ref_free_masked_coder[0], eos_padding=eos, device=0)
                else:
                    patterns, num_bits = table_arrays(name)
                    codes = (pkg.capi.aws_huffman_code * 256)()
                    for s in range(256):
                        codes[s].pattern, codes[s].num_bits = int(patterns[s]), int(num_bits[s])
                    made[key] = pkg.BatchContext(None, eos_padding=eos, device=0, code_table=codes)
        return made[key]

    yield get
    for ctx in made.values():
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# one packed / slotted Huffman call with every array guarded
# ---------------------------------------------------------------------------------------------------------------

STATE = {True: (("overflow_pattern", np.uint32, P32), ("overflow_num_bits", np.uint8, P8)),
         False: (("leftover_working_bits", np.uint64, P64), ("leftover_num_bits", np.uint8, P8))}
ITEM_ARRAYS = (("out_lens", np.uint64, P64), ("status", np.int32, P32), ("consumed", np.uint64, P64))


def huffman_call(ctx, st, encode, data, offs, cap, in_phase, out_phase, fill, slots=None, caps=None, out_init=None):
    """Runs aws_huffman_{en,de}code_batch_device with every array guarded. Returns (results, launches): the arrays
    as the call left them, after their guards and the inputs were checked."""
    n = len(offs) - 1
    inputs = {"in_": place(data, in_phase, fill), "in_offsets": place(np.asarray(offs, np.uint64), P64)}
    if caps is not None:
        inputs["out_offsets"] = place(np.asarray(slots, np.uint64), P64)
        inputs["out_caps"] = place(np.asarray(caps, np.uint64), P64)
    outputs = {"out": place(canary(cap) if out_init is None else out_init, out_phase)}
    if caps is None:
        outputs["out_offsets"] = scratch_array(np.uint64, n + 1, P64)
    for key, dtype, phase in ITEM_ARRAYS + STATE[encode]:
        outputs[key] = scratch_array(dtype, n, phase)
    fn = "aws_huffman_%s_batch_device" % ("encode" if encode else "decode")
    count = launches(ctx, lambda: ctx._call(fn, n, {**inputs, **outputs}, cap, stream=st.cuda_stream,
                                           in_size=int(offs[-1])))
    res = {k: p.read("%s %s" % (fn, k)) for k, p in outputs.items()}
    for k, p in inputs.items():
        res[k] = p.read("%s %s" % (fn, k), unchanged=True)
    return res, count


def assert_packed(got, want, cap, what):
    """Offsets and per-item arrays always equal the oracle's (with all the room it needs); the payload only when
    the capacity holds it."""
    for key in want:
        if key != "out":
            bad = np.flatnonzero(np.asarray(got[key]) != np.asarray(want[key]))
            assert not len(bad), "%s: %s differs at %s (got %s, want %s)" % (
                what, key, bad[:5].tolist(), np.asarray(got[key])[bad[:3]], np.asarray(want[key])[bad[:3]])
    need = int(want["out_offsets"][-1])
    if need <= cap:
        bad = np.flatnonzero(got["out"][:need] != want["out"][:need])
        assert not len(bad), "%s: payload differs at byte %s" % (what, bad[:5].tolist())


def short_strings(rng, table, n=1500):
    data, offs = refcodec.random_batch(rng, n, 0, 200, table)
    return data, offs


# route: (tables, input maker, launches, (in phase, out phase) pairs). Launches as counted in encode_on_device
# (csrc/huffman_batch.cu) with the per-item arrays asked for:
#   string encoder: str_prep/bits/scan/pack 4 (:343), its gated tiled redo tile_index_kernel 1 (:376) and
#                   encode_tiled_kernel<true> 1 (:382), fill_packed_meta_kernel 1 (:409)
#   slots encoder:  launch_scan 1 (:244), slot_tile_index_kernel 1 (:259), encode_slots_kernel 1 (:279), meta 1
#   tiled:          tile_index_kernel + encode_tiled_kernel<true> 2 (n > 1) or encode_tiled_kernel<false> 1, meta 1
#   generic:        encode_items_warp_kernel<false> 1 (:421), launch_scan 1, encode_items_warp_kernel<true> 1 (:426)
ENCODE_ROUTES = {
    "strings": (("hpack", "test"), short_strings, 7, ALIGNED_IN),
    "slots": (("hpack", "test"), lambda rng, t: refcodec.random_batch(rng, 40, 2049, 6000, t), 4, ALIGNED_IN),
    "tiled_batch": (("hpack", "test"), short_strings, 3, SHIFTED_IN),
    "tiled_single": (("hpack", "test"), lambda rng, t: refcodec.random_batch(rng, 1, 20000, 20000, t), 2,
                     ALIGNED_IN + SHIFTED_IN),
    # a symbol without a code (the masked coder) or a 32-bit code: the generic per-item encoder
    "generic_masked": (("masked",), lambda rng, t: refcodec.random_batch(rng, 500, 0, 100, "test", zipf=False), 3,
                       ALIGNED_IN + SHIFTED_IN),
    "generic_max32": (("max32",), lambda rng, t: batch(rng, "max32", rng.integers(0, 200, size=500), "zipf"), 3,
                      ALIGNED_IN + SHIFTED_IN),
}


@pytest.mark.parametrize("route", list(ENCODE_ROUTES))
def test_packed_encode_routes(contexts, tables, oracle, stream, route):
    names, make, want_launches, pairs = ENCODE_ROUTES[route]
    rng = np.random.default_rng(0xE1 + list(ENCODE_ROUTES).index(route))
    inputs = {name: make(rng, name) for name in names}
    combos = list(itertools.product(names, (0xFF, 0x5A)))
    # every phase pair at every capacity; table, padding and neighbour fill rotate so that they meet every capacity
    for k, ((in_phase, out_phase), cap_kind) in enumerate(itertools.product(pairs, CAPACITIES)):
        name, eos = combos[(k + k // 4) % len(combos)]
        fill = FILLS[k % 3]
        data, offs = inputs[name]
        want = oracle.encode_batch(tables(name), eos, data, offs, 4 * len(data) + 64)
        cap = capacity(cap_kind, int(want["out_offsets"][-1]))
        what = "%s %s eos=%#x phases=%d/%d fill=%s cap=%s" % (route, name, eos, in_phase, out_phase, fill, cap_kind)
        got, count = huffman_call(contexts(name, eos), stream, True, data, offs, cap, in_phase, out_phase, fill)
        assert count == want_launches, "%s: %d launches" % (what, count)
        assert_packed(got, want, cap, what)


# decode routes: batch decoder decode_batch_kernel<false> 1 (:472); generic decode_items_thread_kernel<false> 1
# (:568), launch_scan 1, decode_items_thread_kernel<true> 1 (:573)
DECODE_ROUTES = {
    "batch": (("hpack", "test"), None, 1),
    "generic_lut8208": (("lut8208",), None, 3),
    "generic_forced": (("hpack", "test"), "AWS_HUFFMAN_BATCH_FORCE_GENERIC", 3),
}


@pytest.mark.parametrize("route", list(DECODE_ROUTES))
def test_packed_decode_routes(contexts, tables, oracle, stream, route):
    names, switch, want_launches = DECODE_ROUTES[route]
    rng = np.random.default_rng(0xD1 + list(DECODE_ROUTES).index(route))
    payloads = {}
    for name in names:
        if name in ("hpack", "test"):
            data, offs = short_strings(rng, name)
        else:
            data, offs = batch(rng, name, rng.integers(0, 200, size=1500), "uniform")
        enc = oracle.encode_batch(tables(name), 0xFF, data, offs, 4 * len(data) + 64)
        clean = enc["out"][:int(enc["out_offsets"][-1])].copy()
        payloads[name] = (clean, flip_bits(rng, clean), enc["out_offsets"])
    for k, ((in_phase, out_phase), cap_kind) in enumerate(itertools.product(ALIGNED_IN + SHIFTED_IN, CAPACITIES)):
        name = names[(k + k // 4) % len(names)]
        fill = FILLS[k % 3]
        clean, flipped, offs = payloads[name]
        payload = clean if (k + k // 4) // len(names) % 2 == 0 else flipped
        want = oracle.decode_batch(tables(name), payload, offs, 8 * len(payload) + 64)
        cap = capacity(cap_kind, int(want["out_offsets"][-1]))
        what = "%s %s phases=%d/%d fill=%s cap=%s" % (route, name, in_phase, out_phase, fill, cap_kind)
        got, count = huffman_call(contexts(name, 0xFF, switch), stream, False, payload, offs, cap, in_phase, out_phase,
                                  fill)
        assert count == want_launches, "%s: %d launches" % (what, count)
        assert_packed(got, want, cap, what)


# ---- one long stream: the chunk grid shifted by the input's lead ---------------------------------------------------

CHUNK = 128  # bytes of a 1024-bit chunk of the stream decoder
STREAM_CHUNKS = 520  # 66,560 B: above the 64 KiB at which one item takes the stream kernels


def stream_payloads(rng, oracle, table, lengths):
    """{length: {kind: payload}} for clean streams (symbols with codes of at most 8 bits, so that every length is
    reached exactly, padded with ones), streams cut mid-code, corrupted streams and arbitrary bytes."""
    patterns, num_bits = refcodec.table_arrays("hpack")
    short = np.flatnonzero((num_bits > 0) & (num_bits <= 8)).astype(np.uint8)
    sampler = refcodec.zipf_symbol_sampler(num_bits)
    data = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=120_000)])
    data = np.where(np.isin(data, short), data, short[0]).astype(np.uint8)
    enc = oracle.encode_batch(table, 0xFF, data, [0, len(data)], 4 * len(data) + 64)
    full = enc["out"][:int(enc["out_offsets"][-1])]
    ends = np.cumsum(num_bits[data].astype(np.int64))  # bit position after each symbol
    mixed = np.ascontiguousarray(sampler[rng.integers(0, 65536, size=120_000)])
    enc = oracle.encode_batch(table, 0xFF, mixed, [0, len(mixed)], 4 * len(mixed) + 64)
    cut_source = enc["out"][:int(enc["out_offsets"][-1])]
    noise = with_runs(rng, rng.integers(0, 256, size=max(lengths) + 16, dtype=np.uint8))
    out = {}
    for length in lengths:
        m = int(np.searchsorted(ends, 8 * length, side="right"))
        assert ends[m - 1] > 8 * (length - 1)
        clean = full[:length].copy()
        free = 8 * length - int(ends[m - 1])
        if free:
            clean[-1] |= (1 << free) - 1
        broken = flip_bits(rng, clean, every=20_000)
        where = int(rng.integers(0, length - 6)) if length % 2 else length - 6
        broken[where:where + 6] = 0xFF  # 48 one-bits: no code
        out[length] = {"clean": clean, "cut": cut_source[:length].copy(), "corrupt": broken,
                       "bytes": noise[:length].copy()}
    return out


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "multi_kernel"])
def test_stream_decode_at_every_lead(contexts, tables, oracle, stream, fused):
    """Every lead 0..15 of the input, with lead + length at -1, 0, +1..+5 and +127 bytes from a multiple of the
    128-byte chunk (the last chunk absorbs a tail of fewer than 32 bits). Launches (decode_stream_fast): the fused
    kernel and its verify 2 (:525), sync, fix x2, verify, repair, counts 6 (:541), launch_scan 1, write 1 (:545)."""
    ctx = contexts("hpack", 0xFF, None if fused else "AWS_HUFFMAN_BATCH_NO_FUSED_STREAM")
    table = tables("hpack")
    rng = np.random.default_rng(0x5F + fused)
    deltas = (-1, 0, 1, 2, 3, 4, 5, 127)
    cases = [(lead, CHUNK * STREAM_CHUNKS + d - lead) for lead in range(16) for d in deltas]
    payloads = stream_payloads(rng, oracle, table, sorted({length for _, length in cases}))
    k = 0
    for lead, length in cases:
        for kind, payload in payloads[length].items():
            offs = np.array([0, length], dtype=np.uint64)
            want = oracle.decode_batch(table, payload, offs, 8 * length + 64)
            out_phase, fill, cap_kind = (3 * lead + k) % 16, FILLS[k % 3], CAPACITIES[k % 4]
            k += 1
            cap = capacity(cap_kind, int(want["out_offsets"][-1]))
            what = "%s lead=%d len=%d out phase=%d fill=%s cap=%s" % (kind, lead, length, out_phase, fill, cap_kind)
            got, count = huffman_call(ctx, stream, False, payload, offs, cap, lead, out_phase, fill)
            assert count == (10 if fused else 8), "%s: %d launches" % (what, count)
            assert_packed(got, want, cap, what)
            if kind == "clean":
                assert int(want["status"][0]) == OK and int(want["consumed"][0]) == length, what


# ---- slotted layout ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("encode", [True, False], ids=["encode", "decode"])
def test_slotted_layout_on_the_device(contexts, tables, oracle, stream, encode):
    """Capacities scattered around the need (some items come back SHORT_BUFFER); the output starts as canary bytes
    and every byte outside the bytes an item wrote is still canary. One launch: the per-item kernel's writing pass
    (encode_items_warp_kernel<true>, decode_items_thread_kernel<true>)."""
    rng = np.random.default_rng(0x51 + encode)
    for k, (name, (in_phase, out_phase)) in enumerate(zip(("hpack", "test") * 2, [(0, 0), (3, 5), (8, 1), (15, 15)])):
        table = tables(name)
        data, offs = short_strings(rng, name, 1200)
        eos = (0xFF, 0x5A)[k % 2] if encode else 0xFF
        enc = oracle.encode_batch(table, eos, data, offs, 4 * len(data) + 64)
        if encode:
            need = enc["out_lens"]
        else:
            data, offs = enc["out"][:int(enc["out_offsets"][-1])].copy(), enc["out_offsets"]
            if k % 2:
                data = flip_bits(rng, data)
            need = oracle.decode_batch(table, data, offs, 8 * len(data) + 64)["out_lens"]
        slots, caps, total = slots_around(rng, need, -8 if encode else -6, 3)
        out_init = canary(total)
        run = oracle.encode_batch if encode else oracle.decode_batch
        want = run(*((table, eos) if encode else (table,)), data, offs, total, out_offsets=slots, out_caps=caps,
                   out=out_init.copy())
        what = "%s phases=%d/%d" % (name, in_phase, out_phase)
        got, count = huffman_call(contexts(name, eos), stream, encode, data, offs, total, in_phase, out_phase,
                                  FILLS[k % 3], slots=slots, caps=caps, out_init=out_init)
        assert count == 1, "%s: %d launches" % (what, count)
        for key in want:
            if key != "out":
                assert np.array_equal(got[key], want[key]), "%s: %s differs at %s" % (
                    what, key, np.flatnonzero(np.asarray(got[key]) != np.asarray(want[key]))[:5])
        bad = np.flatnonzero(got["out"] != want["out"])
        assert not len(bad), "%s: out differs at byte %s" % (what, bad[:5].tolist())
        assert (want["status"] == SHORT_BUFFER).any() and (want["status"] == OK).any(), what


# ---- streaming continuation with the state kept on the device ------------------------------------------------------

def resume_round(ctx, st, encode, chunks, cap, in_phase, out_phase, state, fill):
    """One *_resume_device call over every stream: chunk i into a slot of `cap` bytes; `state` (two Placed arrays)
    is read and updated in place by the call."""
    n = len(chunks)
    data = np.concatenate([np.asarray(c, np.uint8) for c in chunks]) if sum(map(len, chunks)) else np.zeros(0, np.uint8)
    offs = offsets([len(c) for c in chunks])
    arrays = {"in_": place(data, in_phase, fill), "in_offsets": place(offs, P64),
              "out_offsets": place(np.arange(n, dtype=np.uint64) * cap, P64),
              "out_caps": place(np.full(n, cap, np.uint64), P64), "out": place(canary(n * cap), out_phase)}
    for key, dtype, phase in ITEM_ARRAYS:
        arrays[key] = scratch_array(dtype, n, phase)
    keys = [key for key, _, _ in STATE[encode]]
    fn = "aws_huffman_%s_batch_resume_device" % ("encode" if encode else "decode")
    ctx._call(fn, n, {**arrays, keys[0]: state[0], keys[1]: state[1]}, n * cap, stream=st.cuda_stream,
              in_size=len(data))
    got = {k: arrays[k].read("%s %s" % (fn, k), unchanged=k in ("in_", "in_offsets", "out_offsets", "out_caps"))
           for k in arrays}
    got[keys[0]], got[keys[1]] = state[0].read(fn + " state"), state[1].read(fn + " state")
    return got


@pytest.mark.parametrize("table_name", ["test", "hpack"])
@pytest.mark.parametrize("cap", [1, 3])
def test_resume_encode_device_with_output_in_pieces(contexts, tables, oracle, stream, table_name, cap):
    """test_gpu_resume's output-in-pieces case on device arrays at odd phases, every stream in every call (a finished
    one with nothing left to encode), the overflow state kept on the device."""
    rng = np.random.default_rng(2000 + cap)
    table, ctx = tables(table_name), contexts(table_name)
    n = 129
    texts, offs = refcodec.random_batch(rng, n=n, min_len=0, max_len=90, table=table_name)
    streams = [texts[int(offs[i]):int(offs[i + 1])] for i in range(n)]
    encoders = [oracle.new_encoder(table, 0xFF) for _ in range(n)]
    pos = np.zeros(n, dtype=np.int64)
    state = (scratch_array(np.uint32, n, 4), scratch_array(np.uint8, n, 7))
    state[0].buf[state[0].start:state[0].end] = 0
    state[1].buf[state[1].start:state[1].end] = 0
    done = np.zeros(n, dtype=bool)
    rounds = 0
    while not done.all():
        rounds += 1
        assert rounds < 2000
        chunks = [streams[i][pos[i]:] for i in range(n)]
        in_phase, out_phase = SHIFTED_IN[rounds % 4]
        got = resume_round(ctx, stream, True, chunks, cap, in_phase, out_phase, state, FILLS[rounds % 3])
        for i in range(n):
            out = np.zeros(cap, dtype=np.uint8)
            rc, used, olen = oracle.encode_call(encoders[i], chunks[i], out, 0, cap)
            what = "stream %d round %d" % (i, rounds)
            assert (int(got["status"][i]), int(got["consumed"][i]), int(got["out_lens"][i])) == (rc, used, olen), what
            assert np.array_equal(got["out"][i * cap:i * cap + olen], out[:olen]), what
            assert int(got["overflow_num_bits"][i]) == encoders[i].overflow_bits.num_bits, what
            if encoders[i].overflow_bits.num_bits:
                assert int(got["overflow_pattern"][i]) == encoders[i].overflow_bits.pattern, what
            assert rc in (OK, SHORT_BUFFER), what
            pos[i] += used
            done[i] = rc == OK and pos[i] == len(streams[i])
    assert rounds > 1


@pytest.mark.parametrize("table_name", ["test", "hpack"])
@pytest.mark.parametrize("in_chunk,out_cap", [(2, 3), (5, 1)])
def test_resume_decode_device_fed_in_chunks(contexts, tables, oracle, stream, table_name, in_chunk, out_cap):
    """test_gpu_resume's fed-in-chunks case on device arrays at odd phases, every stream in every call, the decoder
    registers kept on the device."""
    rng = np.random.default_rng(177 + in_chunk * 31 + out_cap)
    table, ctx = tables(table_name), contexts(table_name)
    n = 97
    texts, offs = refcodec.random_batch(rng, n=n, min_len=0, max_len=120, table=table_name)
    enc = oracle.encode_batch(table, 0xFF, texts, offs, out_capacity=4 * len(texts) + 16)
    streams = [enc["out"][int(enc["out_offsets"][i]):int(enc["out_offsets"][i + 1])] for i in range(n)]
    decoders = [oracle.new_decoder(table) for _ in range(n)]
    pos = np.zeros(n, dtype=np.int64)
    fed = np.zeros(n, dtype=np.int64)
    done = np.zeros(n, dtype=bool)
    outputs = [[] for _ in range(n)]
    state = (scratch_array(np.uint64, n, 8), scratch_array(np.uint8, n, 5))
    state[0].buf[state[0].start:state[0].end] = 0
    state[1].buf[state[1].start:state[1].end] = 0
    rounds = 0
    while not done.all():
        rounds += 1
        assert rounds < 5000
        for i in range(n):
            if pos[i] == fed[i]:
                fed[i] = min(len(streams[i]), fed[i] + in_chunk)
        chunks = [streams[i][pos[i]:fed[i]] for i in range(n)]
        in_phase, out_phase = SHIFTED_IN[rounds % 4]
        got = resume_round(ctx, stream, False, chunks, out_cap, in_phase, out_phase, state, FILLS[rounds % 3])
        for i in range(n):
            out = np.zeros(out_cap, dtype=np.uint8)
            rc, used, olen = oracle.decode_call(decoders[i], chunks[i], out, 0, out_cap)
            what = "stream %d round %d" % (i, rounds)
            assert (int(got["status"][i]), int(got["consumed"][i]), int(got["out_lens"][i])) == (rc, used, olen), what
            assert np.array_equal(got["out"][i * out_cap:i * out_cap + olen], out[:olen]), what
            assert int(got["leftover_num_bits"][i]) == decoders[i].num_bits, what
            assert int(got["leftover_working_bits"][i]) == decoders[i].working_bits, what
            assert rc in (OK, SHORT_BUFFER), what
            if not done[i]:
                outputs[i].append(out[:olen].copy())
            pos[i] += used
            if rc == OK and fed[i] == len(streams[i]) and pos[i] == fed[i]:
                done[i] = True
    for i in range(n):
        want = texts[int(offs[i]):int(offs[i + 1])]
        have = np.concatenate(outputs[i]) if outputs[i] else np.zeros(0, np.uint8)
        assert np.array_equal(have[:len(want)], want), "stream %d" % i


# ---- encoded lengths ---------------------------------------------------------------------------------------------

def test_encoded_lengths_on_the_device(contexts, tables, oracle, stream):
    """aws_huffman_get_encoded_length_batch_device (one encoded_length_kernel launch) at input phases 0, 1, 7 and 15,
    with empty items mixed in."""
    rng = np.random.default_rng(0x1E)
    for k, in_phase in enumerate((0, 1, 7, 15)):
        name = ("hpack", "test")[k % 2]
        data, offs = refcodec.random_batch(rng, 900, 0, 300, name, zipf=k < 2)
        lens = np.diff(offs.astype(np.int64))
        lens[rng.choice(len(lens), size=100, replace=False)] = 0
        offs = offsets(lens)
        data = data[:int(offs[-1])]
        n = len(lens)
        d_in, d_off = place(data, in_phase, FILLS[k % 3]), place(offs, P64)
        d_lens = scratch_array(np.uint64, n, P64)
        ctx = contexts(name)
        count = launches(ctx, lambda: ctx.encoded_lengths_device(n, d_in, d_off, d_lens, stream=stream.cuda_stream))
        assert count == 1
        got = d_lens.read("lens")
        d_in.read("in", unchanged=True)
        d_off.read("in_offsets", unchanged=True)
        want = [oracle.encoded_length(tables(name), data[int(offs[i]):int(offs[i + 1])]) for i in range(n)]
        assert np.array_equal(got, want), "phase %d: lens differ at %s" % (in_phase, np.flatnonzero(got != want)[:5])


# ---- empty batches -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("fn", ["aws_huffman_encode_batch_device", "aws_huffman_decode_batch_device",
                                "aws_huffman_encode_batch_resume_device", "aws_huffman_decode_batch_resume_device",
                                "aws_hpack_string_encode_batch_device", "aws_hpack_string_decode_batch_device"])
def test_empty_packed_batch_writes_the_first_offset(contexts, stream, fn):
    """n == 0 in the packed layout: out_offsets[0] = 0 is the whole result, as the host calls write it; with
    out_offsets NULL the call still succeeds."""
    ctx = contexts("hpack")
    for null in (False, True):
        d_off = None if null else scratch_array(np.uint64, 1, P64)
        if fn.startswith("aws_hpack"):
            ctx.hpack_device("encode" in fn, 0, None, None, 0, None, 0, d_off, stream=stream.cuda_stream)
        else:
            ctx._call(fn, 0, {"out_offsets": d_off}, 0, stream=stream.cuda_stream)
        if not null:
            assert int(d_off.read(fn + " out_offsets")[0]) == 0


def test_empty_encoded_length_batch(contexts, stream):
    ctx = contexts("hpack")
    assert launches(ctx, lambda: ctx.encoded_lengths_device(0, None, None, None, stream=stream.cuda_stream)) == 0


# ---------------------------------------------------------------------------------------------------------------
# HPACK string literals (aws_hpack_string_{en,de}code_batch_device)
# ---------------------------------------------------------------------------------------------------------------

LITERAL_CAPS = ("need", "need-1", "generous")


def hpack_call(ctx, st, encode, data, offs, cap, in_phase, out_phase, fill, mode=0):
    n = len(offs) - 1
    d_in, d_off = place(data, in_phase, fill), place(np.asarray(offs, np.uint64), P64)
    d_out, d_out_off = place(canary(cap), out_phase), scratch_array(np.uint64, n + 1, P64)
    d_status = None if encode else scratch_array(np.int32, n, P32)
    count = launches(ctx, lambda: ctx.hpack_device(encode, n, d_in, d_off, len(data), d_out, cap, d_out_off,
                                                  status=d_status, mode=mode, stream=st.cuda_stream))
    what = "hpack %s" % ("encode" if encode else "decode")
    d_in.read(what + " in", unchanged=True)
    d_off.read(what + " in_offsets", unchanged=True)
    got = {"out": d_out.read(what + " out"), "out_offsets": d_out_off.read(what + " out_offsets")}
    if d_status is not None:
        got["status"] = d_status.read(what + " status")
    return got, count


def assert_literals(got, want, want_offs, cap, what, want_status=None):
    assert np.array_equal(got["out_offsets"], want_offs), "%s: offsets differ at %s" % (
        what, np.flatnonzero(got["out_offsets"] != want_offs)[:5])
    if want_status is not None:
        assert np.array_equal(got["status"], want_status), "%s: status differs at %s" % (
            what, np.flatnonzero(got["status"] != want_status)[:5])
    if len(want) <= cap:
        assert np.array_equal(got["out"][:len(want)], want), "%s: bytes differ" % what


@pytest.mark.parametrize("mode", [lit.SMALLEST, lit.NEVER, lit.ALWAYS])
def test_hpack_encode_on_the_device(contexts, literal_oracle, stream, mode):
    """Launches: with a Huffman pass the inner encode_on_device takes the string encoder when `in` is aligned (6, no
    per-item arrays) and the tiled kernel otherwise (2); then hpack_plan_kernel, launch_scan, hpack_frame_kernel."""
    rng = np.random.default_rng(0x4E + mode)
    ctx = contexts("hpack")
    data, offs = _strings(rng, 600, 200)
    want, want_offs = literal_oracle.encode_batch(data, offs, mode)
    for k, ((in_phase, out_phase), cap_kind) in enumerate(itertools.product(ALIGNED_IN + SHIFTED_IN, LITERAL_CAPS)):
        cap = capacity(cap_kind, len(want))
        what = "mode %d phases=%d/%d cap=%d of %d" % (mode, in_phase, out_phase, cap, len(want))
        got, count = hpack_call(ctx, stream, True, data, offs, cap, in_phase, out_phase, FILLS[k % 3], mode)
        inner = 0 if mode == lit.NEVER else (6 if in_phase == 0 else 2)
        assert count == inner + 3, "%s: %d launches" % (what, count)
        assert_literals(got, want, want_offs, cap, what)


@pytest.mark.parametrize("route", ["one_kernel", "passes"])
def test_hpack_decode_on_the_device(contexts, literal_oracle, stream, monkeypatch, route):
    """one_kernel: decode_batch_kernel<true> alone (1 launch); passes (AWS_HUFFMAN_HPACK_PASSES, read per call):
    parse, launch_scan, move, the batch decoder, finish, launch_scan, move (7). Clean and damaged literals."""
    if route == "passes":
        monkeypatch.setenv("AWS_HUFFMAN_HPACK_PASSES", "1")
    else:
        monkeypatch.delenv("AWS_HUFFMAN_HPACK_PASSES", raising=False)
    rng = np.random.default_rng(0x4D)
    ctx = contexts("hpack")
    data, offs = _strings(rng, 600, 160)
    framed, f_offs = literal_oracle.encode_batch(data, offs, lit.SMALLEST)
    cases = {"clean": (framed, f_offs), "damaged": damaged(rng, framed, f_offs)}
    for k, ((in_phase, out_phase), cap_kind) in enumerate(itertools.product(ALIGNED_IN + SHIFTED_IN, LITERAL_CAPS)):
        label = ("clean", "damaged")[(k + k // 3) % 2]
        f, fo = cases[label]
        want, want_offs, want_status = literal_oracle.decode_batch(f, fo)
        cap = capacity(cap_kind, len(want))
        what = "%s %s phases=%d/%d cap=%d of %d" % (route, label, in_phase, out_phase, cap, len(want))
        got, count = hpack_call(ctx, stream, False, f, fo, cap, in_phase, out_phase, FILLS[k % 3])
        assert count == (1 if route == "one_kernel" else 7), "%s: %d launches" % (what, count)
        assert_literals(got, want, want_offs, cap, what, want_status)
        if label == "damaged":
            assert set(want_status.tolist()) > {lit.OK}, what


def test_hpack_one_long_literal_on_the_device(contexts, literal_oracle, stream):
    """One 400 KB literal: encode on the tiled kernel (n == 1), decode on the passes route with its host read-back of
    the payload size and the stream kernels (parse, scan, move, 10 stream launches, finish, scan, move)."""
    rng = np.random.default_rng(0x400)
    ctx = contexts("hpack")
    data, offs = refcodec.random_batch(rng, 1, 400_000, 400_000, "hpack")
    framed, f_offs = literal_oracle.encode_batch(data, offs, lit.SMALLEST)
    for in_phase, out_phase, cap in ((0, 7, len(framed)), (9, 0, len(framed) - 1)):
        got, count = hpack_call(ctx, stream, True, data, offs, cap, in_phase, out_phase, "echo", lit.SMALLEST)
        assert count == 4, count
        assert_literals(got, framed, f_offs, cap, "encode phases=%d/%d cap=%d" % (in_phase, out_phase, cap))
    want, want_offs, want_status = literal_oracle.decode_batch(framed, f_offs)
    for in_phase, out_phase, cap in ((0, 0, len(want)), (13, 3, len(want) - 1), (5, 11, len(want) // 2)):
        got, count = hpack_call(ctx, stream, False, framed, f_offs, cap, in_phase, out_phase, "ones")
        assert count == 16, count
        assert_literals(got, want, want_offs, cap, "decode phases=%d/%d cap=%d" % (in_phase, out_phase, cap),
                        want_status)
    assert int(want_status[0]) == lit.OK and np.array_equal(want, data)


# ---------------------------------------------------------------------------------------------------------------
# caller streams
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("encode", [True, False], ids=["encode", "decode"])
def test_calls_follow_the_caller_stream(pkg, coders, oracle, oracle_tables, encode):
    """On a side stream, with no host synchronisation until the end: a sleep, then the copies that produce the
    input, then the call, which must read the input the stream wrote. Then a small call and one about 100 times
    larger on the same fresh context, so its scratch buffers grow between them: the first call's results must be
    intact at the end."""
    import torch
    dev = torch.device("cuda", 0)
    table = oracle_tables["hpack"]
    rng = np.random.default_rng(0xCA11 + encode)
    ctx = pkg.BatchContext(coders.coder("hpack"), eos_padding=0xFF, device=0)
    try:
        jobs = []
        for n in (60, 60, 6000):
            data, offs = refcodec.random_batch(rng, n, 0, 200, "hpack")
            want = oracle.encode_batch(table, 0xFF, data, offs, 4 * len(data) + 64)
            if not encode:
                data, offs = want["out"][:int(want["out_offsets"][-1])].copy(), want["out_offsets"]
                want = oracle.decode_batch(table, data, offs, 8 * len(data) + 64)
            src = (torch.from_numpy(data).to(dev), torch.from_numpy(offs.view(np.int64)).to(dev))
            cap = int(want["out_offsets"][-1]) + 64
            dst = {"in_": torch.zeros(len(data) + 1, dtype=torch.uint8, device=dev)[1:],
                   "in_offsets": torch.zeros(n + 1, dtype=torch.int64, device=dev),
                   "out": torch.zeros(cap, dtype=torch.uint8, device=dev),
                   "out_offsets": torch.zeros(n + 1, dtype=torch.int64, device=dev),
                   "out_lens": torch.zeros(n, dtype=torch.int64, device=dev),
                   "status": torch.full((n,), -1, dtype=torch.int32, device=dev)}
            jobs.append((src, dst, want, len(data), cap))
        torch.cuda.synchronize(dev)
        side = torch.cuda.Stream(dev)
        fn = ctx.encode_device if encode else ctx.decode_device
        with torch.cuda.stream(side):
            for j, (src, dst, want, size, cap) in enumerate(jobs):
                if j == 0:
                    torch.cuda._sleep(100_000_000)  # tens of milliseconds
                dst["in_"].copy_(src[0])
                dst["in_offsets"].copy_(src[1])
                fn(len(src[1]) - 1, dst, size, cap, stream=side.cuda_stream)
        side.synchronize()
        for j, (src, dst, want, size, cap) in enumerate(jobs):
            total = int(want["out_offsets"][-1])
            what = "call %d" % j
            assert np.array_equal(dst["out_offsets"].cpu().numpy().view(np.uint64), want["out_offsets"]), what
            assert np.array_equal(dst["out_lens"].cpu().numpy().view(np.uint64), want["out_lens"]), what
            assert np.array_equal(dst["status"].cpu().numpy(), want["status"]), what
            assert np.array_equal(dst["out"][:total].cpu().numpy(), want["out"][:total]), what
    finally:
        ctx.close()
