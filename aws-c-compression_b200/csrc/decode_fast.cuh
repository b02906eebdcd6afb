// Fast decode paths for the packed layout.
//
//   decode_batch_kernel        batches of independent short strings (BASELINE configs 2, 5): one thread
//                              per string, persistent blocks with the whole decode LUT in shared memory.
//                              SINGLE PASS: every string is decoded once into a private shared-memory
//                              row; a block scan and a single-pass decoupled look-back give every string
//                              its output offset; the rows are moved into a dense shared-memory image of
//                              the tile's output, which leaves with coalesced 128-bit stores.
//
//   stream_fused_kernel        one long stream (BASELINE config 4), SINGLE PASS: chunked speculative decode
//                              that exploits Huffman self-synchronisation. The stream is cut into fixed
//                              chunks of kChunkBits; each thread starts kPrerollBits before its chunk at
//                              an arbitrary bit, and by the time it reaches its chunk it is (almost
//                              always) on a true code boundary; it then decodes its chunk into its row
//                              and records where it entered, where it left and how many symbols it saw.
//                              A chunk is confirmed when it entered exactly where its predecessor left;
//                              the few that are not are decoded again from the right spot. Output as above.
//
//   stream_sync/fix/verify/    the multi-kernel form of the same idea (correct for ANY prefix code,
//   repair/counts/write        self-synchronising or not): the fallback behind the fused kernel's fail flag.
//
//   decode_span_smem           the decode step both single-pass kernels share (register-resident stream
//                              cursor, branch-free predicated rounds, two symbols per lookup).
//
// Termination rules, status, cursor position and leftover register follow the reference loop
// (source/huffman.c:230-281, refill :196-211); see SURVEY.md App. B.6/B.7 for the closed forms.
#pragma once

#include "device_common.cuh"

namespace hb {

#ifndef HB_ROWCOPY_BATCH
#define HB_ROWCOPY_BATCH 1
#endif
#ifndef HB_DEC_UNIFIED_STEPS
#define HB_DEC_UNIFIED_STEPS 6
#endif
constexpr int kUnifiedSteps = HB_DEC_UNIFIED_STEPS;

constexpr uint32_t kDecLutMaxSmem = 8192;  // entries (32 KiB); larger tables use the generic kernels

// Full lookup of one window (device LUT format: device_common.cuh). Returns a leaf entry or 0 (hole);
// callers that want one symbol at a time use dlut_len1 / dlut_sym1 of the result.
__device__ __forceinline__ uint32_t dec_walk(const uint32_t *s_lut, uint32_t root_bits, uint32_t window, uint32_t e) {
    uint32_t used = root_bits;
    while (e != 0 && !dlut_is_leaf(e)) {
        const uint32_t width = dlut_link_width(e);
        e = s_lut[dlut_link_base(e) + ((window << used) >> (32 - width))];
        used += width;
    }
    return e;
}
__device__ __forceinline__ uint32_t dec_lookup(const uint32_t *s_lut, uint32_t root_bits, uint32_t window) {
    const uint32_t e = s_lut[window >> (32 - root_bits)];
    return dlut_is_leaf(e) ? e : dec_walk(s_lut, root_bits, window, e);
}

enum : uint32_t {
    kTermStop = 0,     // reached the caller's stop position (more stream follows)
    kTermEnd = 1,      // the stream ended (all bits used, padding, or a code cut short): SUCCESS
    kTermUnknown = 2,  // a window with >= 32 bits left matched no code: UNKNOWN_SYMBOL
};

struct DecodeSpan {
    uint64_t pos;   // bit position after the last decoded symbol
    uint64_t nsym;  // symbols decoded
    uint32_t term;
};

// Big-endian bit reader over global memory using aligned 32-bit loads; zero beyond `end_byte`.
struct BitReader {
    const uint32_t *wp;     // next aligned word to load
    const uint32_t *wlast;  // aligned word holding the last valid byte
    uint32_t last_mask;     // keeps the valid leading bytes of *wlast (big-endian value)
    uint64_t buf;           // unread bits, left-aligned
    int nb;                 // how many bits of buf came from loaded words

    __device__ __forceinline__ uint32_t load_word() {
        uint32_t w = 0;
        if (wp <= wlast) {
            w = __byte_perm(__ldg(wp), 0, 0x0123);
            if (wp == wlast) w &= last_mask;
        }
        ++wp;
        return w;
    }
    __device__ __forceinline__ void init(const uint8_t *base, uint64_t bit_pos, uint64_t end_byte) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(base) + (bit_pos >> 3);
        const uintptr_t e = reinterpret_cast<uintptr_t>(base) + end_byte;  // one past the last valid byte
        wp = reinterpret_cast<const uint32_t *>(a & ~uintptr_t(3));
        if (end_byte == 0 || e <= (a & ~uintptr_t(3))) {
            wlast = wp - 1;  // nothing valid from here on
            last_mask = 0;
        } else {
            wlast = reinterpret_cast<const uint32_t *>((e - 1) & ~uintptr_t(3));
            const uint32_t valid = (uint32_t)(e - reinterpret_cast<uintptr_t>(wlast));  // 1..4
            last_mask = 0xffffffffu << (8 * (4 - valid));
        }
        const uint32_t lead = (uint32_t)(8 * (a & 3) + (bit_pos & 7));
        const uint32_t w = load_word();
        buf = (uint64_t)w << (32 + lead);
        nb = 32 - (int)lead;
    }
    __device__ __forceinline__ void refill() {
        if (nb <= 32) {
            buf |= (uint64_t)load_word() << (32 - nb);
            nb += 32;
        }
    }
    __device__ __forceinline__ uint32_t window() const { return (uint32_t)(buf >> 32); }
    __device__ __forceinline__ void consume(uint32_t n) {
        buf <<= n;
        nb -= (int)n;
    }
};

// Packs symbols into aligned 32-bit global stores (byte stores only for a ragged head or tail).
struct ByteWriter {
    uint8_t *wordp;   // aligned address of the word being assembled
    uint32_t pack;
    uint32_t count;   // bytes already in `pack` (including the skipped head bytes)
    uint32_t head;    // bytes at the front of the first word that are not ours
    uint64_t room;    // bytes we may still write

    __device__ __forceinline__ void init(uint8_t *out, uint64_t out_room) {
        const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(out) & 3);
        wordp = out - mis;
        pack = 0;
        count = mis;
        head = mis;
        room = out_room;
    }
    __device__ __forceinline__ void flush_partial(uint32_t upto) {
        for (uint32_t i = head; i < upto; ++i) {
            if (room) {
                wordp[i] = (uint8_t)(pack >> (8 * i));
                --room;
            }
        }
    }
    __device__ __forceinline__ void put(uint32_t sym) {
        pack |= (sym & 0xffu) << (8 * count);
        if (++count == 4) {
            if (head == 0 && room >= 4) {
                *reinterpret_cast<uint32_t *>(wordp) = pack;
                room -= 4;
            } else {
                flush_partial(4);
            }
            head = 0;
            wordp += 4;
            pack = 0;
            count = 0;
        }
    }
    __device__ __forceinline__ void finish() {
        if (count > head) flush_partial(count);
    }
};

// Decodes from bit `start` while the position is below `stop` (<= end_bit = 8 * end_byte).
// kSkipHoles: pre-roll policy — a hole just advances one bit (we are only hunting for a boundary).
template <bool kWrite, bool kSkipHoles>
__device__ __forceinline__ DecodeSpan decode_span(
    const uint32_t *s_lut, uint32_t root_bits, const uint8_t *base, uint64_t start, uint64_t stop, uint64_t end_byte,
    ByteWriter *writer) {
    const uint64_t end_bit = end_byte * 8;
    DecodeSpan r;
    r.pos = start;
    r.nsym = 0;
    r.term = kTermStop;
    if (start >= stop) {
        if (start >= end_bit) r.term = kTermEnd;
        return r;
    }
    BitReader br;
    br.init(base, start, end_byte);
    uint64_t pos = start;
    uint64_t nsym = 0;
    while (true) {
        br.refill();
        const uint32_t e = dec_lookup(s_lut, root_bits, br.window());
        const uint64_t bits_left = end_bit - pos;
        if (e == 0) {
            if (kSkipHoles) {
                if (bits_left <= 1) { r.term = kTermEnd; break; }
                br.consume(1);
                pos += 1;
                if (pos >= stop) break;
                continue;
            }
            r.term = bits_left < 32 ? kTermEnd : kTermUnknown;
            break;
        }
        const uint32_t used = dlut_len1(e);
        if (used > bits_left) { r.term = kTermEnd; break; }
        br.consume(used);
        pos += used;
        ++nsym;
        if (kWrite) writer->put(dlut_sym1(e));
        if (pos >= stop) {
            if (pos >= end_bit) r.term = kTermEnd;
            break;
        }
    }
    r.pos = pos;
    r.nsym = nsym;
    return r;
}

// decoder->working_bits / num_bits and the cursor position after a call that emitted `cbits` bits of
// symbols from an item of `len` bytes (fresh decoder). SURVEY.md App. B.7.
__device__ __forceinline__ void leftover_state(
    const uint8_t *item, uint64_t len, uint64_t cbits, bool stopped_early, uint64_t *consumed, uint64_t *working,
    uint8_t *num_bits) {
    uint64_t pulled = len;
    if (stopped_early) {
        const uint64_t need = (cbits + 32 + 7) >> 3;
        pulled = need < len ? need : len;
    }
    const uint64_t first = cbits >> 3;
    uint64_t reg = 0;
    for (uint64_t i = first; i < pulled && i < first + 8; ++i) reg |= (uint64_t)item[i] << (56 - 8 * (i - first));
    reg <<= (cbits & 7);
    if (consumed) *consumed = pulled;
    if (working) *working = reg;
    if (num_bits) *num_bits = (uint8_t)(pulled * 8 - cbits);
}

// ---------------------------------------------------------------------------------------------
// Position-based decode from shared memory.
//
// The encoded bytes of a tile are staged in shared memory as BIG-ENDIAN 32-bit words, so the next 32
// stream bits at bit position `pos` are one funnel shift of two neighbouring words — no bit register
// to refill, no branches in the common case: window = funnel(word[pos/32], word[pos/32 + 1], pos%32).
// kPadded: the stream layout of decode_stream_*: every 32-word chunk row is followed by a copy of the
// next row's first word (row stride 33 words), which keeps lanes that sit at the same offset of
// different chunks on different banks.
// ---------------------------------------------------------------------------------------------
template <bool kPadded>
__device__ __forceinline__ uint32_t smem_window(const uint32_t *s_in, uint32_t pos) {
    const uint32_t idx = kPadded ? (pos >> 5) + (pos >> 10) : (pos >> 5);
    return __funnelshift_l(s_in[idx + 1], s_in[idx], pos);
}

// Packs symbols into aligned 32-bit global stores; one PRMT per symbol, byte stores only for the
// first and last partial word of the span.
struct WordWriter {
    uint8_t *base;   // out + off rounded down to 4 bytes
    uint32_t phase;  // off & 3
    uint32_t k;      // phase + symbols so far
    uint32_t pack;
    uint64_t room;   // bytes that may be written from `out + off`

    __device__ __forceinline__ void init(uint8_t *out, uint64_t out_room) {
        phase = (uint32_t)(reinterpret_cast<uintptr_t>(out) & 3);
        base = out - phase;
        k = phase;
        pack = 0;
        room = out_room;
    }
    // shifts in symbol 1 (kSecond = false) or symbol 2 (kSecond = true) of a LUT leaf entry
    template <bool kSecond>
    __device__ __forceinline__ void put(uint32_t entry) {
        pack = __byte_perm(pack, entry, kSecond ? 0x6321 : 0x5321);
        ++k;
        if ((k & 3u) == 0) {
            const uint32_t done = k - phase;  // symbols so far
            if (k == 4 && phase != 0) {
                // first word is shared with the previous span: only our bytes
                for (uint32_t i = phase; i < 4; ++i)
                    if (i - phase < room) base[i] = (uint8_t)(pack >> (8 * i));
            } else if (done <= room) {
                *reinterpret_cast<uint32_t *>(base + k - 4) = pack;
            } else {
                for (uint32_t i = 0; i < 4; ++i)
                    if (done - 4 + i < room) base[k - 4 + i] = (uint8_t)(pack >> (8 * i));
            }
        }
    }
    __device__ __forceinline__ void finish() {
        const uint32_t tail = k & 3u;  // symbols waiting in `pack` (its top `tail` bytes)
        if (tail == 0) return;
        const uint32_t first = (k < 4) ? phase : 0u;  // the span never completed a word
        const uint32_t word0 = k - tail;              // byte offset of the open word from `base`
        for (uint32_t i = first; i < tail; ++i) {
            const uint64_t sym_index = (uint64_t)(word0 + i) - phase;
            if (sym_index < room) base[word0 + i] = (uint8_t)(pack >> (8 * (4 - tail + i)));
        }
    }
};

struct SpanS {
    uint32_t pos;   // stage-relative bit position after the last decoded symbol
    uint32_t nsym;
    uint32_t term;
};

// Decodes from stage bit `pos` until `stop`; the stream itself ends at `end` (stop <= end; both are
// stage-relative bit positions). Same rules as decode_span.
template <bool kWrite, bool kPadded, bool kSkipHoles, typename Writer = WordWriter>
__device__ __forceinline__ SpanS decode_smem(
    const uint32_t *s_in, const uint32_t *s_lut, uint32_t root_bits, uint32_t pos, uint32_t stop, uint32_t end,
    Writer *writer) {
    SpanS r;
    uint32_t nsym = 0;
    uint32_t term = kTermStop;
    // fast region: at least 32 real bits follow `pos`, so a match can never lean on the zero fill and a
    // hole is an error straight away
    const uint32_t fast_end = (end >= 32u) ? min(stop, end - 31u) : 0u;
    // two symbols per lookup while even the second one is sure to start before `stop`.
    // Codes longer than the root index (a few % of symbols) need a walk through sub-tables. Doing that
    // walk the moment one lane needs it would make the other 31 lanes wait almost every iteration, so
    // a lane that hits a link parks (`pending`) and parked lanes are resolved together every few steps.
    const uint32_t pair_end = fast_end > root_bits ? fast_end - root_bits : 0u;
    constexpr int kStepsPerRound = 6;
    bool pending = false;
    while (pos < pair_end) {
#pragma unroll
        for (int step = 0; step < kStepsPerRound; ++step) {
            if (!pending && pos < pair_end) {
                const uint32_t e = s_lut[smem_window<kPadded>(s_in, pos) >> (32 - root_bits)];
                if (dlut_is_leaf(e)) {
                    pos += dlut_total_len(e);
                    nsym += dlut_count(e);
                    if (kWrite) {
                        writer->template put<false>(e);
                        if (dlut_count(e) == 2) writer->template put<true>(e);
                    }
                } else {
                    pending = true;
                }
            }
        }
        if (pending) {
            pending = false;
            const uint32_t window = smem_window<kPadded>(s_in, pos);
            const uint32_t e = dec_walk(s_lut, root_bits, window, s_lut[window >> (32 - root_bits)]);
            if (e == 0) {
                if (kSkipHoles) {
                    ++pos;
                    continue;
                }
                term = kTermUnknown;
                break;
            }
            pos += dlut_len1(e);
            ++nsym;
            if (kWrite) writer->template put<false>(e);
        }
    }
    // one symbol per lookup up to the end of the fast region
    while (term == kTermStop && pos < fast_end) {
        const uint32_t e = dec_lookup(s_lut, root_bits, smem_window<kPadded>(s_in, pos));
        if (e == 0) {
            if (kSkipHoles) {
                ++pos;
                continue;
            }
            term = kTermUnknown;
            break;
        }
        pos += dlut_len1(e);
        ++nsym;
        if (kWrite) writer->template put<false>(e);
    }
    if (term == kTermStop && pos < stop) {
        // fewer than 32 bits of stream remain: the window is the stream zero-extended
        while (true) {
            const uint32_t left = end - pos;
            if (left == 0) { term = kTermEnd; break; }
            const uint32_t window = smem_window<kPadded>(s_in, pos) & (0xffffffffu << (32 - left));
            const uint32_t e = dec_lookup(s_lut, root_bits, window);
            if (e == 0) {
                if (kSkipHoles && left > 1) {
                    ++pos;
                    if (pos >= stop) break;
                    continue;
                }
                term = kTermEnd;  // fewer than 32 bits left: treated as padding (huffman.c:240-244)
                break;
            }
            const uint32_t used = dlut_len1(e);
            if (used > left) { term = kTermEnd; break; }
            pos += used;
            ++nsym;
            if (kWrite) writer->template put<false>(e);
            if (pos >= stop) {
                if (pos >= end) term = kTermEnd;
                break;
            }
        }
    } else if (term == kTermStop && pos >= end) {
        term = kTermEnd;
    }
    r.pos = pos;
    r.nsym = nsym;
    r.term = term;
    return r;
}

// ---------------------------------------------------------------------------------------------
// The hot loop of the single-pass decoders: two symbols per lookup straight from the staged stream,
// symbols emitted as bytes into the thread's shared-memory row. Hand-tightened (shared-window
// addresses, PTX loads/stores) because this loop is most of the decode time:
//   * a lane that meets a code longer than the root index (a link) spends its NEXT step on the sub-table the
//     link names, with its position unchanged: every step is one lookup, whatever the table
//   * both symbol bytes of an entry are always stored and the address advances by the entry's count:
//     no branch; a one-symbol entry leaves a stray byte that the next store overwrites (rows have room
//     for one byte more than they can hold)
// Runs while at least 32 + root_bits real bits follow `pos`; the caller finishes the span with
// decode_smem (one symbol per lookup, end-of-stream rules).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u8(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// The stream words under the cursor live in registers: w0 holds bit `pos`, w1 the word after it, w2 is
// fetched one word ahead, so the dependent chain of a step is funnel -> LUT load -> add and the stream
// loads are off it. A span never leaves its padded row in here (the callers' spans end at a row boundary,
// or fewer than 32 bits after one), so the words are consecutive in shared memory.
// kRaw: the stage holds the stream's bytes as they are in memory (a bulk copy put them there: decode_batch_kernel with
// HB_DEC_TMA_STAGE); a word is byte-swapped when it is fetched.
template <bool kRaw>
struct StreamCursorT {
    uint32_t w0, w1, w2;
    uint32_t wa;  // shared-window address of the word after w2
    int limit;    // first bit position after w0
    __device__ __forceinline__ static uint32_t fetch(uint32_t addr) {
        const uint32_t v = lds_u32(addr);
        return kRaw ? __byte_perm(v, 0, 0x0123) : v;
    }
    template <bool kPadded>
    __device__ __forceinline__ void init(uint32_t in_addr, uint32_t pos) {
        wa = in_addr + (kPadded ? (pos >> 5) + (pos >> 10) : (pos >> 5)) * 4;
        w0 = fetch(wa);
        w1 = fetch(wa + 4);
        w2 = fetch(wa + 8);
        wa += 12;
        limit = (int)((pos | 31u) + 1u);
    }
    __device__ __forceinline__ uint32_t window(uint32_t pos) const { return __funnelshift_l(w1, w0, pos); }
    // after `pos` moved forward by at most 32 bits
    __device__ __forceinline__ void follow(uint32_t pos) {
        if ((int)pos >= limit) {
            w0 = w1;
            w1 = w2;
            w2 = fetch(wa);
            wa += 4;
            limit += 32;
        }
    }
};
using StreamCursor = StreamCursorT<false>;

// Decodes stage bits from `pos` until `stop`; the stream itself ends at `end` (stop <= end; stage-relative
// bit positions). Same rules and results as decode_smem (which follows the reference loop); symbols go
// to the shared-memory row at out_addr when kEmit. nsym is only meaningful when emitting.
template <bool kEmit, bool kPadded, bool kSkipHoles>
__device__ __forceinline__ SpanS decode_span_smem(
    const uint32_t *s_in, const uint32_t *s_lut, uint32_t root_bits, uint32_t pos, uint32_t stop, uint32_t end,
    uint32_t out_addr) {
    constexpr uint32_t kParked = 0x80000000u;  // positions are far below 2^31: a parked lane fails "pos < pair_end"
    const uint32_t out0 = out_addr;
    SpanS r;
    r.term = kTermStop;
    if (pos < stop) {
        // two symbols per lookup while at least 32 real bits follow and even the second symbol is sure to
        // start before `stop`
        const uint32_t fast_end = (end >= 32u) ? min(stop, end - 31u) : 0u;
        const uint32_t pair_end = fast_end > root_bits ? fast_end - root_bits : 0u;
        const uint32_t in_addr = (uint32_t)__cvta_generic_to_shared(s_in);
        uint32_t lut_addr = (uint32_t)__cvta_generic_to_shared(s_lut);
        // (opaque copy: otherwise the compiler re-derives the base from the shared window in every step)
        asm volatile("mov.u32 %0, %0;" : "+r"(lut_addr));
        const uint32_t shift = 32 - root_bits;
        StreamCursor c;
        c.init<kPadded>(in_addr, pos);
        // Every step is ONE table lookup, whatever the table: a lane whose lookup returned a link (a code
        // longer than the root index: a few % of the symbols) keeps its position and spends its next step
        // on the sub-table the link names, while the other lanes carry on with their own symbols. No lane
        // ever waits for another lane's long code and there is no separate walk.
        //   {tbase, tshift, tused}: table to index, its index shift, window bits the upper levels consumed
        uint32_t tbase = lut_addr, tshift = shift, tused = 0;
        while (pos < pair_end) {
#pragma unroll
            for (int step = 0; step < kUnifiedSteps; ++step) {
                const uint32_t e = lds_u32(tbase + (((c.window(pos) << tused) >> tshift) << 2));
                const bool active = pos < pair_end;
                const bool leaf = dlut_is_leaf(e);
                const bool adv = active && leaf;
                const bool link = active && !leaf && e != 0u;
                const bool hole = active && e == 0u;
                // (inactive lanes are always in the root state: a lane only leaves the span on a leaf or a hole)
                tused = link ? tused + 32u - tshift : 0u;
                tshift = link ? 32u - (e >> 20) : shift;
                tbase = link ? lut_addr + ((e & 0xFFFFFu) << 2) : lut_addr;
                if (adv) pos += e >> 24;
                if (hole) {
                    if (kSkipHoles) ++pos;
                    else pos |= kParked;  // >= 32 real bits and no code matches: UNKNOWN_SYMBOL, the lane stops here
                }
                if (kEmit) {
#ifndef HB_ABL_NO_EMIT  // (timing-only ablations: HB_ABL_* builds give wrong results on purpose)
                    const uint32_t on = adv ? 1u : 0u;
                    asm volatile(
                        "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\t@p st.shared.u8 [%0], %1;\n\t@p st.shared.u8 [%0+1], %2;\n\t}" ::"r"(out_addr),
                        "r"(e >> 8), "r"(e >> 16), "r"(on)
                        : "memory");
#endif
                    if (adv) out_addr += e & 3u;
                }
                const bool cross = (adv || (kSkipHoles && hole)) && (int)pos >= c.limit;
                if (cross) {
                    c.w0 = c.w1;
                    c.w1 = c.w2;
                    c.limit += 32;
                }
                {
                    const uint32_t on = cross ? 1u : 0u;
                    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p ld.shared.u32 %0, [%1];\n\t}"
                                 : "+r"(c.w2)
                                 : "r"(c.wa), "r"(on));
                }
                if (cross) c.wa += 4;
            }
        }
        if (pos & kParked) {
            pos &= ~kParked;
            r.term = kTermUnknown;
        }
        // the last few symbols of the span: one lookup at a time with the end-of-stream rules (the window is
        // the stream zero-extended, huffman.c:196-211; a code that does not fit ends the stream, :240-255).
        // A two-symbol entry still counts when its second code starts before `stop` and ends inside the stream.
        while (r.term == kTermStop && pos < stop) {
            const uint32_t left = end - pos;  // >= 1
            uint32_t window = c.window(pos);
            if (left < 32u) window &= 0xffffffffu << (32u - left);
            uint32_t e = lds_u32(lut_addr + ((window >> shift) << 2));
            if (e != 0 && !dlut_is_leaf(e)) e = dec_walk(s_lut, root_bits, window, e);
            if (e == 0) {
                if (kSkipHoles && left > 1u) {
                    ++pos;
                    c.follow(pos);
                    continue;
                }
                r.term = left < 32u ? kTermEnd : kTermUnknown;  // fewer than 32 bits left: padding
                break;
            }
            const uint32_t len1 = dlut_len1(e);
            if (len1 > left) {
                r.term = kTermEnd;  // a code cut short by the end of the stream
                break;
            }
            const bool two = dlut_count(e) == 2u && pos + len1 < stop && dlut_total_len(e) <= left;
            if (kEmit) {
                sts_u8(out_addr, e >> 8);
                if (two) sts_u8(out_addr + 1, e >> 16);
                out_addr += two ? 2u : 1u;
            }
            pos += two ? dlut_total_len(e) : len1;
            c.follow(pos);
        }
    }
    if (r.term == kTermStop && pos >= end) r.term = kTermEnd;
    r.pos = pos;
    r.nsym = out_addr - out0;
    return r;
}

// ---------------------------------------------------------------------------------------------
// The LEAN decode step (round 2): the same walk over the same tables, re-encoded as 64-bit entries ("LUT2",
// built in huffman_batch.cu from the 32-bit LUT) so that a step needs no selects and no per-table state
// machine:
//     x  [7:0] symbol 1   [15:8] symbol 2   [21:16] length of symbol 1's code from the symbol's first bit
//        [31:30] symbols in the entry (0: link or hole)
//     y  [31:24] bits this step consumes   [23:5] shared-memory address of the table the NEXT step indexes
//        (32-byte aligned)   [4:0] 32 - index width of that table
// A leaf sends the lane back to the root table, a link to its sub-table — after consuming the index bits of the
// level it was found in, so the next step indexes the sub-table with the bits that follow (sub-table leaves
// consume what is left of the code). Whatever the entry is, a step is: funnel, shift by y (the hardware takes
// the low five bits), one multiply-add for the address, one 64-bit load, `pos += y >> 24`, two byte stores,
// `out += x >> 30`, the cursor refill. 20 instructions against 37 of the unified step of round 1.
// A hole (no code matches) leads to a trap table whose entries consume nothing; trapped lanes are noticed
// once per round and the whole span is then decoded again by the exact one-symbol loop below, which also
// finishes every span (end-of-stream rules of huffman.c:196-211, 240-255).
// ---------------------------------------------------------------------------------------------
struct Lut2 {
    uint32_t addr;     // shared-window address of entry 0 (32-byte aligned)
    uint32_t root_ns;  // y of "next step: root table" = addr | (32 - root_bits)
    uint32_t trap_tb;  // table address of the trap table
};

// copies the table into shared memory, turning table offsets into shared-window addresses
__device__ __forceinline__ Lut2 lut2_load(uint2 *s_lut2, const uint2 *g_lut2, uint32_t count, uint32_t root_bits, uint32_t trap_base) {
    Lut2 t;
    t.addr = (uint32_t)__cvta_generic_to_shared(s_lut2);
    t.root_ns = t.addr | (32u - root_bits);
    t.trap_tb = t.addr + 8u * trap_base;
    for (uint32_t i = threadIdx.x; i < count; i += blockDim.x) {
        uint2 e = g_lut2[i];
        e.y += t.addr;
        s_lut2[i] = e;
    }
    return t;
}

struct Lut2Hit {
    uint32_t x;      // entry (0: no code matches the window)
    uint32_t total;  // bits of the whole entry (one or two codes)
};
// exact lookup of one window (one symbol at a time callers use len1 / symbol 1 of x)
__device__ __forceinline__ Lut2Hit lut2_lookup(const Lut2 &t, uint32_t window) {
    uint32_t ns = t.root_ns, used = 0;
    Lut2Hit h;
    while (true) {
        const uint32_t tb = ns & 0x00ffffe0u;
        const uint32_t idx = (window << used) >> (ns & 31u);
        uint32_t x, y;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(x), "=r"(y) : "r"(tb + 8u * idx));
        const uint32_t adv = y >> 24;
        if (x >> 30) {
            h.x = x;
            h.total = used + adv;
            return h;
        }
        if (adv == 0) {
            h.x = 0;
            h.total = 0;
            return h;
        }
        used += adv;
        ns = y;
    }
}
__device__ __forceinline__ uint32_t lut2_len1(uint32_t x) { return (x >> 16) & 63u; }

template <bool kEmit, bool kPadded, bool kSkipHoles, bool kRaw = false>
__device__ __forceinline__ SpanS decode_span_lean(
    const uint32_t *s_in, const Lut2 &t, uint32_t root_bits, uint32_t pos, uint32_t stop, uint32_t end, uint32_t out_addr) {
    constexpr uint32_t kParked = 0x80000000u;
    const uint32_t out0 = out_addr, pos0 = pos;
    SpanS r;
    r.term = kTermStop;
    if (pos < stop) {
        const uint32_t fast_end = (end >= 32u) ? min(stop, end - 31u) : 0u;
        const uint32_t pair_end = fast_end > root_bits ? fast_end - root_bits : 0u;
        const uint32_t in_addr = (uint32_t)__cvta_generic_to_shared(s_in);
        StreamCursorT<kRaw> c;
        c.template init<kPadded>(in_addr, pos);
        uint32_t ns = t.root_ns, tb = t.addr;
        const uint32_t root_tb = t.addr;
        uint32_t acc = 0;  // (kEmit) symbols not stored yet: the low out_addr & 3 bytes
#ifdef HB_PHASE_TIMING
        const long long tl0 = clock64();
        uint32_t rounds = 0;
#endif
#ifndef HB_NO_BULK_ROUNDS
        // Bulk rounds: a step consumes at most max(root_bits, 8) bits (a root entry, or one level of an 8-bit
        // sub-table), so while a whole round is sure to start all its steps before pair_end no step needs the
        // "still inside the span" predicate: two compares and a move less per step (33 -> 30 instructions; the decode
        // step is bound by the ALU pipe, which takes one warp instruction every two cycles).
        {
            const uint32_t step_max = max(root_bits, 8u);
            const uint32_t bulk_end = pair_end > kUnifiedSteps * step_max ? pair_end - kUnifiedSteps * step_max : 0u;
            while (pos < bulk_end) {
#ifdef HB_PHASE_TIMING
                ++rounds;
#endif
#pragma unroll
                for (int step = 0; step < kUnifiedSteps; ++step) {
                    if (kEmit) {

#define HB_STEP_ASM(SWAP) asm volatile( \
                            "{\n\t" \
                            ".reg .pred c, w;\n\t" \
                            ".reg .b32 win, idx, adr, x, u, t, sh, lo, sp, no, wadr;\n\t" \
                            "shf.l.wrap.b32 win, %2, %1, %0;\n\t" \
                            "shf.r.wrap.b32 idx, win, 0, %7;\n\t" \
                            "mad.lo.u32 adr, idx, 8, %8;\n\t" \
                            "ld.shared.v2.u32 {x, %7}, [adr];\n\t" \
                            "and.b32 %8, %7, 0x00ffffe0;\n\t" \
                            "shr.u32 u, %7, 24;\n\t" \
                            "add.u32 %0, %0, u;\n\t" \
                            "and.b32 t, x, 0xffff;\n\t" \
                            "shl.b32 sh, %6, 3;\n\t" \
                            "shf.l.wrap.b32 lo, 0, t, sh;\n\t" \
                            "shf.l.wrap.b32 sp, t, 0, sh;\n\t" \
                            "or.b32 lo, lo, %9;\n\t" \
                            "shr.u32 u, x, 30;\n\t" \
                            "add.u32 no, %6, u;\n\t" \
                            "xor.b32 u, no, %6;\n\t" \
                            "and.b32 u, u, 4;\n\t" \
                            "setp.ne.u32 w, u, 0;\n\t" \
                            "and.b32 wadr, %6, 0xfffffffc;\n\t" \
                            "@w st.shared.u32 [wadr], lo;\n\t" \
                            "selp.b32 %9, sp, lo, w;\n\t" \
                            "mov.b32 %6, no;\n\t" \
                            "setp.ge.s32 c, %0, %5;\n\t" \
                            "@c mov.b32 %1, %2;\n\t" \
                            "@c mov.b32 %2, %3;\n\t" \
                            "@c ld.shared.u32 %3, [%4];\n\t" SWAP \
                            "@c add.u32 %4, %4, 4;\n\t" \
                            "@c add.s32 %5, %5, 32;\n\t" \
                            "}" \
                            : "+r"(pos), "+r"(c.w0), "+r"(c.w1), "+r"(c.w2), "+r"(c.wa), "+r"(c.limit), "+r"(out_addr), "+r"(ns), "+r"(tb), "+r"(acc) \
                            : \
                            : "memory");
                        if (kRaw) { HB_STEP_ASM("@c prmt.b32 %3, %3, 0, 0x0123;\n\t") } else { HB_STEP_ASM("") }
#undef HB_STEP_ASM

                    } else {

#define HB_STEP_ASM(SWAP) asm volatile( \
                            "{\n\t" \
                            ".reg .pred c;\n\t" \
                            ".reg .b32 win, idx, adr, x, u;\n\t" \
                            "shf.l.wrap.b32 win, %2, %1, %0;\n\t" \
                            "shf.r.wrap.b32 idx, win, 0, %6;\n\t" \
                            "mad.lo.u32 adr, idx, 8, %7;\n\t" \
                            "ld.shared.v2.u32 {x, %6}, [adr];\n\t" \
                            "and.b32 %7, %6, 0x00ffffe0;\n\t" \
                            "shr.u32 u, %6, 24;\n\t" \
                            "add.u32 %0, %0, u;\n\t" \
                            "setp.ge.s32 c, %0, %5;\n\t" \
                            "@c mov.b32 %1, %2;\n\t" \
                            "@c mov.b32 %2, %3;\n\t" \
                            "@c ld.shared.u32 %3, [%4];\n\t" SWAP \
                            "@c add.u32 %4, %4, 4;\n\t" \
                            "@c add.s32 %5, %5, 32;\n\t" \
                            "}" \
                            : "+r"(pos), "+r"(c.w0), "+r"(c.w1), "+r"(c.w2), "+r"(c.wa), "+r"(c.limit), "+r"(ns), "+r"(tb) \
                            : \
                            : "memory");
                        if (kRaw) { HB_STEP_ASM("@c prmt.b32 %3, %3, 0, 0x0123;\n\t") } else { HB_STEP_ASM("") }
#undef HB_STEP_ASM

                    }
                }
                if (tb == t.trap_tb) {  // no code matches: leave the loops, the exact loop below redoes the span
                    pos |= kParked;
                    tb = root_tb;
                }
            }
        }
#endif
        while (pos < pair_end || tb != root_tb) {
#ifdef HB_PHASE_TIMING
            ++rounds;
#endif
#pragma unroll
            for (int step = 0; step < kUnifiedSteps; ++step) {
                if (kEmit) {
                    // symbols are collected in `acc` (little-endian, out & 3 bytes pending) and leave as whole
                    // 32-bit words: a quarter of the stores of the byte-by-byte version, and those were 40 % of the
                    // kernel's shared-memory wavefronts (the decode phase is bound by them, not by issue slots)

#define HB_STEP_ASM(SWAP) asm volatile( \
                        "{\n\t" \
                        ".reg .pred p, c, w;\n\t" \
                        ".reg .b32 win, idx, adr, x, u, t, sh, lo, sp, no, wadr;\n\t" \
                        "setp.lt.u32 p, %0, %10;\n\t" \
                        "setp.ne.or.u32 p, %8, %11, p;\n\t" \
                        "shf.l.wrap.b32 win, %2, %1, %0;\n\t" \
                        "shf.r.wrap.b32 idx, win, 0, %7;\n\t" \
                        "mad.lo.u32 adr, idx, 8, %8;\n\t" \
                        "mov.b32 x, 0;\n\t" \
                        "@p ld.shared.v2.u32 {x, %7}, [adr];\n\t" \
                        "and.b32 %8, %7, 0x00ffffe0;\n\t" \
                        "shr.u32 u, %7, 24;\n\t" \
                        "@p add.u32 %0, %0, u;\n\t" \
                        "and.b32 t, x, 0xffff;\n\t" \
                        "shl.b32 sh, %6, 3;\n\t" \
                        "shf.l.wrap.b32 lo, 0, t, sh;\n\t" \
                        "shf.l.wrap.b32 sp, t, 0, sh;\n\t" \
                        "or.b32 lo, lo, %9;\n\t" \
                        "shr.u32 u, x, 30;\n\t" \
                        "add.u32 no, %6, u;\n\t" \
                        "xor.b32 u, no, %6;\n\t" \
                        "and.b32 u, u, 4;\n\t" \
                        "setp.ne.u32 w, u, 0;\n\t" \
                        "and.b32 wadr, %6, 0xfffffffc;\n\t" \
                        "@w st.shared.u32 [wadr], lo;\n\t" \
                        "selp.b32 %9, sp, lo, w;\n\t" \
                        "mov.b32 %6, no;\n\t" \
                        "setp.ge.s32 c, %0, %5;\n\t" \
                        "@c mov.b32 %1, %2;\n\t" \
                        "@c mov.b32 %2, %3;\n\t" \
                        "@c ld.shared.u32 %3, [%4];\n\t" SWAP \
                        "@c add.u32 %4, %4, 4;\n\t" \
                        "@c add.s32 %5, %5, 32;\n\t" \
                        "}" \
                        : "+r"(pos), "+r"(c.w0), "+r"(c.w1), "+r"(c.w2), "+r"(c.wa), "+r"(c.limit), "+r"(out_addr), "+r"(ns), "+r"(tb), "+r"(acc) \
                        : "r"(pair_end), "r"(root_tb) \
                        : "memory");
                    if (kRaw) { HB_STEP_ASM("@c prmt.b32 %3, %3, 0, 0x0123;\n\t") } else { HB_STEP_ASM("") }
#undef HB_STEP_ASM

                } else {

#define HB_STEP_ASM(SWAP) asm volatile( \
                        "{\n\t" \
                        ".reg .pred p, c;\n\t" \
                        ".reg .b32 win, idx, adr, x, u;\n\t" \
                        "setp.lt.u32 p, %0, %8;\n\t" \
                        "setp.ne.or.u32 p, %7, %9, p;\n\t" \
                        "shf.l.wrap.b32 win, %2, %1, %0;\n\t" \
                        "shf.r.wrap.b32 idx, win, 0, %6;\n\t" \
                        "mad.lo.u32 adr, idx, 8, %7;\n\t" \
                        "@p ld.shared.v2.u32 {x, %6}, [adr];\n\t" \
                        "and.b32 %7, %6, 0x00ffffe0;\n\t" \
                        "shr.u32 u, %6, 24;\n\t" \
                        "@p add.u32 %0, %0, u;\n\t" \
                        "setp.ge.s32 c, %0, %5;\n\t" \
                        "@c mov.b32 %1, %2;\n\t" \
                        "@c mov.b32 %2, %3;\n\t" \
                        "@c ld.shared.u32 %3, [%4];\n\t" SWAP \
                        "@c add.u32 %4, %4, 4;\n\t" \
                        "@c add.s32 %5, %5, 32;\n\t" \
                        "}" \
                        : "+r"(pos), "+r"(c.w0), "+r"(c.w1), "+r"(c.w2), "+r"(c.wa), "+r"(c.limit), "+r"(ns), "+r"(tb) \
                        : "r"(pair_end), "r"(root_tb) \
                        : "memory");
                    if (kRaw) { HB_STEP_ASM("@c prmt.b32 %3, %3, 0, 0x0123;\n\t") } else { HB_STEP_ASM("") }
#undef HB_STEP_ASM

                }
            }
            if (tb == t.trap_tb) {  // no code matches: leave the loop, the exact loop below redoes the span
                pos |= kParked;
                tb = root_tb;
            }
        }
#ifdef HB_PHASE_TIMING
        {   // the lane of the warp that ran longest: its rounds and the cycles the warp spent in the loop
            const uint32_t mx = __reduce_max_sync(__activemask(), rounds);
            if (rounds == mx && mx > 0 && kEmit && !kPadded) {
                atomicAdd(&hb_phase_cycles[14], (unsigned long long)(clock64() - tl0));
                atomicAdd(&hb_phase_cycles[15], (unsigned long long)mx);
            }
        }
#endif
        if (pos & kParked) {
            pos = pos0;
            out_addr = out0;
            c.template init<kPadded>(in_addr, pos);
        } else if (kEmit && (out_addr & 3u)) {  // (the bytes above the symbols in `acc` are spare: rows have slack)
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(out_addr & ~3u), "r"(acc) : "memory");
        }
        // the rest of the span (or all of it, after a trap): one lookup at a time with the end-of-stream rules (the
        // window is the stream zero-extended, huffman.c:196-211; a code that does not fit ends the stream,
        // :240-255). A two-symbol entry still counts when its second code starts before `stop` and ends inside
        // the stream.
        while (r.term == kTermStop && pos < stop) {
            const uint32_t left = end - pos;  // >= 1
            uint32_t window = c.window(pos);
            if (left < 32u) window &= 0xffffffffu << (32u - left);
            const Lut2Hit h = lut2_lookup(t, window);
            if (h.x == 0) {
                if (kSkipHoles && left > 1u) {
                    ++pos;
                    c.follow(pos);
                    continue;
                }
                r.term = left < 32u ? kTermEnd : kTermUnknown;  // fewer than 32 bits left: padding
                break;
            }
            const uint32_t len1 = lut2_len1(h.x);
            if (len1 > left) {
                r.term = kTermEnd;  // a code cut short by the end of the stream
                break;
            }
            const bool two = (h.x >> 30) == 2u && pos + len1 < stop && h.total <= left;
            if (kEmit) {
                sts_u8(out_addr, h.x);
                if (two) sts_u8(out_addr + 1, h.x >> 8);
                out_addr += two ? 2u : 1u;
            }
            pos += two ? h.total : len1;
            c.follow(pos);
        }
    }
    if (r.term == kTermStop && pos >= end) r.term = kTermEnd;
    r.pos = pos;
    r.nsym = out_addr - out0;
    return r;
}

// decode_span (bit reader over global memory) with the shared-memory LUT2: the route of tiles that do not fit the stage
template <bool kWrite>
__device__ __forceinline__ DecodeSpan decode_span_lut2(
    const Lut2 &t, const uint8_t *base, uint64_t start, uint64_t stop, uint64_t end_byte, ByteWriter *writer) {
    const uint64_t end_bit = end_byte * 8;
    DecodeSpan r;
    r.pos = start;
    r.nsym = 0;
    r.term = kTermStop;
    if (start >= stop) {
        if (start >= end_bit) r.term = kTermEnd;
        return r;
    }
    BitReader br;
    br.init(base, start, end_byte);
    uint64_t pos = start, nsym = 0;
    while (true) {
        br.refill();
        const Lut2Hit h = lut2_lookup(t, br.window());
        const uint64_t bits_left = end_bit - pos;
        if (h.x == 0) {
            r.term = bits_left < 32 ? kTermEnd : kTermUnknown;
            break;
        }
        const uint32_t used = lut2_len1(h.x);
        if (used > bits_left) { r.term = kTermEnd; break; }
        br.consume(used);
        pos += used;
        ++nsym;
        if (kWrite) writer->put(h.x & 0xffu);
        if (pos >= stop) {
            if (pos >= end_bit) r.term = kTermEnd;
            break;
        }
    }
    r.pos = pos;
    r.nsym = nsym;
    return r;
}

// ---------------------------------------------------------------------------------------------
// Batch of independent strings
// ---------------------------------------------------------------------------------------------
#ifdef HB_PHASE_TIMING  // (development builds: cycles per phase of decode_batch_kernel, thread 0 of every block)
#define HB_PHASE_MARK(i)                                                   \
    do {                                                                   \
        if (tid == 0) {                                                    \
            const long long now_ = clock64();                              \
            atomicAdd(&hb_phase_cycles[i], (unsigned long long)(now_ - t_phase_)); \
            t_phase_ = now_;                                               \
        }                                                                  \
    } while (0)
#else
#define HB_PHASE_MARK(i) do { } while (0)
#endif

// Worker threads of a team. Seven of the warps decode (HB_DEC_PULL_WARPS below); the others only help in the phases
// around it — string table, sort, scan, rows -> image, copy-out. Measured on the 1M-string batch with 7 pullers:
// 256 / 288 / 320 / 352 / 384 threads: 0.2753 / 0.2752 / 0.2650 / 0.2780 / 0.2695 ms.
#ifndef HB_DEC_THREADS
#define HB_DEC_THREADS 320
#endif
#ifndef HB_DEC_TEAMS
#define HB_DEC_TEAMS 2
#endif
constexpr int kDecThreads = HB_DEC_THREADS;  // worker threads of a team
constexpr int kDecWarps = kDecThreads / 32;
constexpr int kDecBlock = kDecThreads + 32;  // a team: its worker warps + 1 scout warp
constexpr int kDecTeams = HB_DEC_TEAMS;      // teams per block (they share the decode table); 5 named barriers each
// Warps of a team that decode (the others wait at the barrier behind the decode phase, which costs nothing). The
// phase cannot end before the tile's longest string does, so more lanes than the work needs only add contention
// to every step of that string: the warps pull groups of 32 strings, longest first.
// (measured, 1M strings of 8..256 B, 9 groups per tile: 8 / 7 / 6 / 5 pulling warps: 0.291 / 0.285 / 0.290 / 0.298 ms)
#ifndef HB_DEC_PULL_WARPS
#define HB_DEC_PULL_WARPS 7
#endif
constexpr int kDecPullWarps = HB_DEC_PULL_WARPS;
constexpr uint32_t kDecDone = 0xffffffffu;
#ifndef HB_DEC_ITEMS_PER_TILE
#define HB_DEC_ITEMS_PER_TILE 288
#endif
constexpr int kDecItemsPerTile = HB_DEC_ITEMS_PER_TILE;  // strings per tile at most (9 groups of 32)
// Named barriers (as in encode_tiled.cuh). Workers among themselves: 1. Hand-off of a tile to the scout: 2 + parity
// (workers arrive without waiting, the scout waits). Result of a look-back: 4 + parity (the scout arrives, the
// workers wait).
__device__ __forceinline__ void dec_worker_sync(uint32_t team) { asm volatile("bar.sync %0, %1;" ::"r"(5 * team + 1), "n"(kDecThreads) : "memory"); }
__device__ __forceinline__ void dec_bar_arrive(uint32_t id) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(kDecBlock) : "memory"); }
__device__ __forceinline__ void dec_bar_sync(uint32_t id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(kDecBlock) : "memory"); }
constexpr uint32_t kDecMaxRow = 4096;        // a staged string decodes to at most this many bytes
constexpr uint32_t kDecRowSlack = 8;         // spare bytes per row (alignment, the emitter's look-ahead byte)

// HB_DEC_TMA_STAGE: the tile's encoded bytes come into the stage by ONE bulk copy (cp.async.bulk global -> shared,
// completion on an mbarrier: the TMA unit moves them while the team sorts its strings) instead of the team's own
// 128-bit loads, byte permutes and stores; the stage then holds the bytes as they are in memory and the decoder
// swaps a word when it fetches it (one PRMT per 32 consumed bits). Not for the framed decoder.
#ifndef HB_DEC_TMA_STAGE
#define HB_DEC_TMA_STAGE 1
#endif
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_copy_to_shared(uint32_t dst, const void *src, uint32_t bytes, uint32_t mbar) {
    // (the stage was read and written through the generic proxy by the previous tile)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "HB_MBAR_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra HB_MBAR_WAIT;\n\t"
        "}" ::"r"(mbar), "r"(parity)
        : "memory");
}

struct DecBatchArgs {
    BatchView b;
    const uint32_t *lut;   // 32-bit table in global memory (the rare tiles that do not fit the stage)
    const uint2 *lut2;     // 64-bit entries of the lean step, copied to shared memory
    uint32_t lut2_count;   // entries (a multiple of 4)
    uint32_t lut2_trap;    // first entry of the trap table
    uint32_t root_bits;
    uint32_t min_len;      // shortest code: a string of L bytes decodes to at most 8 L / min_len symbols
    uint32_t stage_words;  // capacity of the input stage
    uint32_t rows_bytes;   // capacity of the row area
    uint64_t *tile_state;
    uint32_t *ticket;
    uint32_t num_tiles;
    uint32_t items_per_tile;  // <= kDecItemsPerTile, a multiple of 32: fewer when the strings are long, so that a
                              // tile of average strings still fits the stage
};

// Whole team: copies n bytes of a dense image in shared memory (`src` 16-byte aligned, with >= 32 readable bytes
// after n) to `dst` (any alignment) with 128-bit stores.
__device__ __forceinline__ void smem_copy_out(const uint8_t *src, uint8_t *dst, uint32_t n, uint32_t tid, uint32_t nthreads) {
    const uint32_t head = min(n, (16u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15)) & 15u);
    const uint32_t nvec = (n - head) >> 4;
    const uint4 *sv = reinterpret_cast<const uint4 *>(src);
    uint4 *dv = reinterpret_cast<uint4 *>(dst + head);
    const uint32_t tw = head >> 2, r8 = (head & 3u) * 8u;  // the body starts `head` bytes into the image
    for (uint32_t v = tid; v < nvec; v += nthreads) {
        const uint4 a = sv[v], b = sv[v + 1];
        uint32_t w0, w1, w2, w3, w4;
        switch (tw) {  // (uniform)
            case 0: w0 = a.x; w1 = a.y; w2 = a.z; w3 = a.w; w4 = b.x; break;
            case 1: w0 = a.y; w1 = a.z; w2 = a.w; w3 = b.x; w4 = b.y; break;
            case 2: w0 = a.z; w1 = a.w; w2 = b.x; w3 = b.y; w4 = b.z; break;
            default: w0 = a.w; w1 = b.x; w2 = b.y; w3 = b.z; w4 = b.w; break;
        }
        uint4 o;
        o.x = __funnelshift_r(w0, w1, r8);
        o.y = __funnelshift_r(w1, w2, r8);
        o.z = __funnelshift_r(w2, w3, r8);
        o.w = __funnelshift_r(w3, w4, r8);
        dv[v] = o;
    }
    if (tid < head) dst[tid] = src[tid];
    const uint32_t tail0 = head + 16u * nvec;
    if (tid >= 32 && tid - 32 < n - tail0) dst[tail0 + tid - 32] = src[tail0 + tid - 32];
}

// Thread-serial copy of n bytes inside shared memory; src is 4-byte aligned, dst is not.
__device__ __forceinline__ void smem_copy_row(const uint8_t *src, uint8_t *dst, uint32_t n) {
    if (n == 0) return;
    const uint32_t head = min(n, (4u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 3)) & 3u);
    for (uint32_t i = 0; i < head; ++i) dst[i] = src[i];
    const uint32_t body = (n - head) >> 2;  // whole destination words
    if (body) {
        const uint32_t *sw = reinterpret_cast<const uint32_t *>(src);
        uint32_t *dw = reinterpret_cast<uint32_t *>(dst + head);
        const uint32_t sel = 0x3210u + 0x1111u * head;  // bytes head .. head + 3 of a word pair
        uint32_t lo = sw[0];
        uint32_t j = 0;
#if HB_ROWCOPY_BATCH
        // four loads in flight before the four stores (source and destination never overlap within a phase, but
        // the compiler cannot know and would keep every load behind the previous store)
        for (; j + 4 <= body; j += 4) {
            const uint32_t h0 = sw[j + 1], h1 = sw[j + 2], h2 = sw[j + 3], h3 = sw[j + 4];
            dw[j] = __byte_perm(lo, h0, sel);
            dw[j + 1] = __byte_perm(h0, h1, sel);
            dw[j + 2] = __byte_perm(h1, h2, sel);
            dw[j + 3] = __byte_perm(h2, h3, sel);
            lo = h3;
        }
#endif
        for (; j < body; ++j) {
            const uint32_t hi = sw[j + 1];
            dw[j] = __byte_perm(lo, hi, sel);
            lo = hi;
        }
    }
    for (uint32_t i = head + 4 * body; i < n; ++i) dst[i] = src[i];
}

// One thread per string, single pass. Persistent 256-thread blocks, the whole decode LUT in shared
// memory. Per tile of kDecItemsPerTile strings:
//   1. the encoded bytes are staged as big-endian words (coalesced 128-bit loads); strings are SORTED
//      BY LENGTH (counting sort in shared memory) and handed to warps in groups of 32 similar lengths,
//      longest first, warps pulling groups dynamically, so lanes leave the decode loop together
//   2. every string is decoded ONCE; its symbols go byte by byte into a private row of shared memory
//      (row i starts where the string could start at worst: 8 * offset / min_len)
//   3. a block scan of the symbol counts + a single-pass decoupled look-back give every string its
//      output offset
//   4. every thread moves its rows to their final place in a DENSE shared-memory image of the tile's
//      output (laid out with the alignment of its global address), which is then copied out with
//      128-bit coalesced stores. The dense image reuses the input stage and the front of the row area:
//      rows that start in that front part are moved first (their destination lies inside the stage),
//      the others after a barrier (their destination may overlap rows that are already gone).
// A tile whose strings do not fit the stage is decoded straight from global memory in two passes.
// Dynamic shared memory: [LUT][stage words + 2][rows]
// kFramed: the items are HPACK string literals (hpack_literals.cuh): the string table parses each literal's H bit and
// length (the payload is what gets staged / decoded), raw literals are copied instead of decoded, and the padding rule
// of RFC 7541 5.2 is applied to what the decoder leaves over; items with a non-zero status decode to nothing.
// Shared state of one TEAM (8 worker warps + 1 scout warp working on one tile). A block holds kDecTeams teams
// that share ONE copy of the decode table: the table is 38 KB, and what bounds this kernel is the number of
// strings in flight per SM (every phase of a tile is a chain of latencies), so the shared memory a second copy
// would take is worth more as stage and rows.
template <bool kFramed>
struct DecTeamShared {
    uint32_t start[kDecItemsPerTile];   // first bit of the string in the stage
    uint32_t bytes[kDecItemsPerTile];   // encoded length
    uint32_t cnt[kDecItemsPerTile];     // symbols per string
    uint32_t off[kDecItemsPerTile];     // exclusive offsets within the tile
    uint32_t row[kDecItemsPerTile];     // start of the string's row in the row area
    uint16_t perm[kDecItemsPerTile];    // strings in order of decreasing length
    uint8_t flag[kFramed ? kDecItemsPerTile : 4];  // framed: bit 0 raw payload, bit 1 malformed literal
    uint32_t hist[256];
    uint64_t warp_sum[kDecWarps];
    uint32_t tile, next, fits, total;
    uint32_t hand_tile[2];                 // workers -> scout, by hand-off parity
    uint64_t hand_prefix[2];               // scout -> workers
    uint64_t mbar;                         // HB_DEC_TMA_STAGE: completion of the stage's bulk copy
};

template <bool kFramed>
__global__ void __launch_bounds__(kDecTeams * kDecBlock, 1) decode_batch_kernel(DecBatchArgs a) {
    extern __shared__ __align__(128) uint32_t s_lut[];  // [LUT2][team 0: stage, rows][team 1: stage, rows]
    __shared__ DecTeamShared<kFramed> s_teams[kDecTeams];
    static_assert(kDecItemsPerTile <= 2 * kDecThreads, "the block scan handles two strings per thread");
    const uint32_t team = threadIdx.x / kDecBlock, tid = threadIdx.x - team * kDecBlock;
    DecTeamShared<kFramed> &sh = s_teams[team];
    uint32_t (&s_start)[kDecItemsPerTile] = sh.start;
    uint32_t (&s_bytes)[kDecItemsPerTile] = sh.bytes;
    uint32_t (&s_cnt)[kDecItemsPerTile] = sh.cnt;
    uint32_t (&s_off)[kDecItemsPerTile] = sh.off;
    uint32_t (&s_row)[kDecItemsPerTile] = sh.row;
    uint16_t (&s_perm)[kDecItemsPerTile] = sh.perm;
    auto &s_flag = sh.flag;
    uint32_t (&s_hist)[256] = sh.hist;
    uint64_t (&s_warp_sum)[kDecWarps] = sh.warp_sum;
    uint32_t &s_tile = sh.tile, &s_next = sh.next, &s_fits = sh.fits, &s_total = sh.total;
    uint32_t (&s_hand_tile)[2] = sh.hand_tile;
    uint64_t (&s_hand_prefix)[2] = sh.hand_prefix;
    const uint32_t lut_pad = 2u * a.lut2_count;          // words
    const uint32_t stage_bytes = (a.stage_words + 2) * 4;         // (+2 zero words for the window look-ahead)
    const uint32_t team_bytes = ((stage_bytes + 15u) & ~15u) + a.rows_bytes + 64u;
    uint32_t *s_in = s_lut + lut_pad + team * (team_bytes / 4);
    uint8_t *const s_dense = reinterpret_cast<uint8_t *>(s_in);  // the dense image starts where the stage does
    uint8_t *const s_rows = s_dense + ((stage_bytes + 15u) & ~15u);

    const Lut2 lut2 = lut2_load(reinterpret_cast<uint2 *>(s_lut), a.lut2, a.lut2_count, a.root_bits, a.lut2_trap);
    const uint32_t lane = lane_id(), warp = tid >> 5;
    const BatchView &b = a.b;
    constexpr bool kRaw = HB_DEC_TMA_STAGE != 0 && !kFramed;
    const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&sh.mbar);
    if (kRaw && tid == 0) mbar_init(mbar, 1);
    uint32_t stage_phase = 0;  // parity of the bulk copy the team waits for next
    __syncthreads();  // the LUT is in place
    // ================================ scout =====================================================================
    // The ninth warp resolves where the tile's output starts — the sum of the symbol counts of ALL tiles before it
    // (single-pass decoupled look-back) — WHILE the workers stage, decode and compact the tile: the sum does not
    // need the tile's own count, only its predecessors', and those finish at about the same time (tiles are
    // handed out in order). By the time the dense image is ready the position is normally known, so the image goes
    // straight from shared memory to its final place: no parking in a scratch slot, no second copy (round 1 parked
    // every tile for one tile's time because warp 0 only started the look-back after the decode: 14-25 % of the
    // kernel was the wait for that chain of L2 round trips).
    if (warp == kDecWarps) {
        for (uint32_t h = 0;; ++h) {
            dec_bar_sync(5 * team + 2 + (h & 1));  // the workers took a tile
            const uint32_t t = s_hand_tile[h & 1];
            if (t == kDecDone) return;
#ifdef HB_ABL_DEC_NO_LOOKBACK  // (timing-only ablation: wrong output positions)
            const uint64_t prefix = 0;
#else
            const uint64_t prefix = lookback_exclusive(a.tile_state, t);
#endif
            if (lane == 0) s_hand_prefix[h & 1] = prefix;
            dec_bar_arrive(5 * team + 4 + (h & 1));  // result ready
        }
    }
    // ================================ workers ===================================================================
    uint32_t hand = 0;  // tiles handed to the scout so far
    const uint32_t rows_addr = (uint32_t)__cvta_generic_to_shared(s_rows);

#ifdef HB_PHASE_TIMING
    long long t_phase_ = clock64();
#endif
    uint32_t iter = 0;
    for (;; ++iter) {
        dec_worker_sync(team);  // previous tile fully done (and the LUT is in place on the first trip)
        if (tid == 0) {
            s_tile = atomicAdd(a.ticket, 1u);
            s_next = kDecPullWarps;
            s_fits = 1;
        }
        for (uint32_t i = tid; i < 256; i += kDecThreads) s_hist[i] = 0;
        dec_worker_sync(team);
        const uint32_t tile = s_tile;
        if (tile >= a.num_tiles) break;
        if (tid == 0) s_hand_tile[hand & 1] = tile;
        dec_bar_arrive(5 * team + 2 + (hand & 1));  // the scout starts on the tile's position
        ++hand;
#ifdef HB_PHASE_TIMING
        if (tid == 0 && tile < 8192) hb_tile_times[0][tile] = hb_now_ns();
#endif
        const uint64_t item0 = (uint64_t)tile * a.items_per_tile;
        const uint32_t nitems = (uint32_t)min((uint64_t)a.items_per_tile, b.n - item0);
        const uint32_t ngroups = (nitems + 31) / 32;

        // ---- string table: where each string starts in the stage and in the row area; length histogram -------
        const uint64_t byte0 = b.in_offsets[item0], byte1 = b.in_offsets[item0 + nitems];
        const uintptr_t addr0 = reinterpret_cast<uintptr_t>(b.in) + byte0;
        const uint32_t lead = (uint32_t)(addr0 & 15);  // the stage starts on a 16-byte boundary
        const uint64_t nwords64 = (byte1 - byte0 + lead + 3) >> 2;
        // row i starts at 4 * ceil(2 * offset / min_len) + slack * i: never before the end of row i - 1
        const uint64_t rows_need = 4 * ((2 * (byte1 - byte0) + a.min_len - 1) / a.min_len) + (uint64_t)kDecRowSlack * (nitems + 1);
        bool fits = nwords64 <= a.stage_words && rows_need <= a.rows_bytes;
        // (kRaw) The whole 16-byte pieces of the tile's bytes are requested NOW, as one bulk copy: they arrive while
        // the team builds its string table and sorts. (A tile that turns out to hold a string too long for a row is
        // not decoded from the stage; the copy is awaited all the same.)
        const bool bulk = kRaw && fits && (nwords64 >> 2) != 0;
        if (bulk && tid == 0)
            bulk_copy_to_shared((uint32_t)__cvta_generic_to_shared(s_in), reinterpret_cast<const void *>(addr0 - lead),
                                16u * (uint32_t)(nwords64 >> 2), mbar);
        for (uint32_t it = tid; it < nitems; it += kDecThreads) {
            const uint64_t in0 = b.in_offsets[item0 + it];
            uint64_t len = b.in_offsets[item0 + it + 1] - in0;
            uint64_t skip = 0;  // bytes of the item before its payload
            if (kFramed) {
                uint32_t h, np;
                uint64_t plen;
                const int32_t st = hpack_parse_literal(b.in + in0, len, h, np, plen);
                s_flag[it] = (uint8_t)((st != kStatusOk ? 2u : 0u) | (h ? 0u : 1u));
                if (st != kStatusOk && b.status) b.status[item0 + it] = st;
                len = st == kStatusOk ? plen : 0;
                skip = np;
            }
            s_start[it] = (uint32_t)(in0 + skip - byte0) * 8 + lead * 8;
            s_bytes[it] = (uint32_t)min(len, (uint64_t)0xffffffffu);
            s_row[it] = 4 * (uint32_t)((2 * (in0 - byte0) + a.min_len - 1) / a.min_len) + kDecRowSlack * it;
            if (8 * len / a.min_len + kDecRowSlack > kDecMaxRow) s_fits = 0;
            atomicAdd(&s_hist[255 - (uint32_t)min(len, (uint64_t)255)], 1u);
        }
        dec_worker_sync(team);
        const bool staged = fits && s_fits != 0;
        if (staged) {
            const uint32_t nwords = (uint32_t)nwords64;
            const uint32_t nquads = nwords >> 2;  // whole 128-bit pieces; the ragged end goes word by word
            const uint32_t *gw = reinterpret_cast<const uint32_t *>(addr0 - lead);
            if (kRaw) {
                // ---- (the bulk copy is under way) the ragged end, bytes as they are in memory -------------------------
                for (uint32_t j = 4 * nquads + tid; j < nwords; j += kDecThreads) s_in[j] = __ldg(gw + j);
            } else {
                // ---- stage the tile's encoded bytes as big-endian words -------------------------------------------
                const uint4 *g4 = reinterpret_cast<const uint4 *>(addr0 - lead);
                for (uint32_t j = tid; j < nquads; j += kDecThreads) {
                    const uint4 v = __ldg(g4 + j);
                    uint4 o;
                    o.x = __byte_perm(v.x, 0, 0x0123);
                    o.y = __byte_perm(v.y, 0, 0x0123);
                    o.z = __byte_perm(v.z, 0, 0x0123);
                    o.w = __byte_perm(v.w, 0, 0x0123);
                    reinterpret_cast<uint4 *>(s_in)[j] = o;
                }
                for (uint32_t j = 4 * nquads + tid; j < nwords; j += kDecThreads)
                    s_in[j] = __byte_perm(__ldg(gw + j), 0, 0x0123);
            }
            if (tid < 2) s_in[nwords + tid] = 0;
        }
        if (warp == 0) {
            // exclusive scan of the 256 bins, 8 per lane
            uint32_t v[8], sum = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                v[i] = s_hist[lane * 8 + i];
                sum += v[i];
            }
            uint32_t run = warp_inclusive_scan(sum) - sum;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                s_hist[lane * 8 + i] = run;
                run += v[i];
            }
        }
        dec_worker_sync(team);
        for (uint32_t it = tid; it < nitems; it += kDecThreads) {
            const uint32_t rank = atomicAdd(&s_hist[255 - min(s_bytes[it], 255u)], 1u);
            s_perm[rank] = (uint16_t)it;
        }
        dec_worker_sync(team);

        if (kRaw && bulk) {  // the stage's bytes have landed
            mbar_wait(mbar, stage_phase);
            stage_phase ^= 1u;
        }
        HB_PHASE_MARK(0);  // ticket, string table, staging, sort
        // ---- decode (staged: once, into the rows; otherwise: count) ------------------------------------------
        for (uint32_t g = warp < (uint32_t)kDecPullWarps ? warp : ngroups; g < ngroups;) {
            const uint32_t slot = g * 32 + lane;
            if (slot < nitems) {
                const uint32_t it = s_perm[slot];
                const uint64_t item = item0 + it;
                const uint32_t nbytes = s_bytes[it];
                uint64_t cbits = 0;
                uint32_t nsym = 0, term = kTermEnd;
                const uint32_t flag = kFramed ? s_flag[it] : 0u;
                // (framed: where the payload starts in global memory; s_start holds it relative to the tile)
                const uint8_t *payload = b.in + (kFramed ? byte0 + (s_start[it] >> 3) - lead : b.in_offsets[item]);
                int32_t st = kStatusOk;
                if (kFramed && flag != 0) {
                    if (flag == 1u) {  // raw literal: the payload is the string
                        nsym = nbytes;
                        if (staged) {
                            const uint32_t first = s_start[it] >> 3, row = rows_addr + s_row[it];
                            for (uint32_t k = 0; k < nbytes; ++k)
                                sts_u8(row + k, s_in[(first + k) >> 2] >> (24 - 8 * ((first + k) & 3)));
                        }
                    }
                } else if (staged) {
                    const uint32_t ib = s_start[it], ie = ib + nbytes * 8;
                    const SpanS r = decode_span_lean<true, false, false, kRaw>(s_in, lut2, a.root_bits, ib, ie, ie, rows_addr + s_row[it]);
                    cbits = r.pos - ib;
                    nsym = r.nsym;
                    term = r.term;
                    if (kFramed && term != kTermUnknown) {
                        const uint32_t rem = ie - r.pos;  // what the decoder left over: must be < 8 bits, all ones
                        if (rem >= 8u || (rem != 0u && (smem_window<false>(s_in, r.pos) >> (32u - rem)) != (1u << rem) - 1u))
                            st = kStatusInvalidPadding;
                    }
                } else {
                    const uint64_t len = kFramed ? (uint64_t)nbytes : b.in_offsets[item + 1] - b.in_offsets[item];
                    const DecodeSpan r = decode_span_lut2<false>(lut2, payload, 0, len * 8, len, nullptr);
                    cbits = r.pos;
                    nsym = (uint32_t)r.nsym;
                    term = r.term;
                    if (kFramed && term != kTermUnknown) {
                        uint64_t bits = 0;
                        uint8_t nb = 0;
                        leftover_state(payload, len, cbits, false, nullptr, &bits, &nb);
                        if (!hpack_padding_ok(bits, nb)) st = kStatusInvalidPadding;
                    }
                }
                if (term == kTermUnknown) st = kStatusUnknownSymbol;
                if (kFramed && st != kStatusOk) nsym = 0;  // a literal that fails decodes to nothing
                s_cnt[it] = nsym;
                if (b.status && !(kFramed && (flag & 2u))) b.status[item] = st;
                if (b.consumed || b.leftover_working_bits || b.leftover_num_bits) {
                    const uint64_t in0 = b.in_offsets[item];
                    leftover_state(
                        b.in + in0, b.in_offsets[item + 1] - in0, cbits, term == kTermUnknown,
                        b.consumed ? b.consumed + item : nullptr,
                        b.leftover_working_bits ? b.leftover_working_bits + item : nullptr,
                        b.leftover_num_bits ? b.leftover_num_bits + item : nullptr);
                }
            }
            uint32_t next = 0;
            if (lane == 0) next = atomicAdd(&s_next, 1u);
            g = __shfl_sync(0xffffffffu, next, 0);
        }
        dec_worker_sync(team);

        HB_PHASE_MARK(1);  // decode (to the barrier behind it)
        // ---- offsets: block scan (2 strings per thread); the tile's count goes out at once ------------------------
        const uint32_t par = iter & 1u;
        const uint32_t c0 = 2 * tid < nitems ? s_cnt[2 * tid] : 0u;
        const uint32_t c1 = 2 * tid + 1 < nitems ? s_cnt[2 * tid + 1] : 0u;
        const uint64_t mine = (uint64_t)c0 + c1;
        const uint64_t incl = warp_inclusive_scan64(mine);
        if (lane == 31) s_warp_sum[warp] = incl;
        dec_worker_sync(team);
        if (warp == 0) {
            uint64_t w = lane < kDecWarps ? s_warp_sum[lane] : 0;
            const uint64_t wi = warp_inclusive_scan64(w);
            if (lane < kDecWarps) s_warp_sum[lane] = wi - w;
            const uint64_t total = __shfl_sync(0xffffffffu, wi, kDecWarps - 1);
            if (lane == 0) {
                lookback_publish_aggregate(a.tile_state, tile, total);
                s_total = (uint32_t)total;
#ifdef HB_PHASE_TIMING
                if (tile < 8192) hb_tile_times[1][tile] = hb_now_ns();
#endif
            }
        }
        dec_worker_sync(team);
        {
            const uint64_t e0 = s_warp_sum[warp] + (incl - mine);  // exclusive, within the tile
            if (2 * tid < nitems) {
                s_off[2 * tid] = (uint32_t)e0;
                if (b.out_lens) b.out_lens[item0 + 2 * tid] = c0;
            }
            if (2 * tid + 1 < nitems) {
                s_off[2 * tid + 1] = (uint32_t)(e0 + c0);
                if (b.out_lens) b.out_lens[item0 + 2 * tid + 1] = c1;
            }
            if (tid == 0) s_next = kDecWarps;
        }
        dec_worker_sync(team);
        const uint32_t total = s_total;

        HB_PHASE_MARK(2);  // scan, publish
        if (staged) {
            // rows -> dense image at the front of the stage area. Rows that start before `front` lie where the
            // image may grow: they go first (their destination ends inside the stage area); the host sizes the
            // areas so that the image ends before row offset `front`
            const uint32_t front = stage_bytes > kDecMaxRow + 32 ? ((stage_bytes - kDecMaxRow - 32) & ~3u) : 0u;
#pragma unroll 1
            for (int phase = 0; phase < 2; ++phase) {
                for (uint32_t it = tid; it < nitems; it += kDecThreads) {
                    const uint32_t row = s_row[it];
#ifndef HB_ABL_NO_COPY
                    if ((row < front) == (phase == 0)) smem_copy_row(s_rows + row, s_dense + s_off[it], s_cnt[it]);
#endif
                }
                dec_worker_sync(team);
            }
        }
        HB_PHASE_MARK(3);  // rows -> image
        // ---- where the tile goes: the scout has been summing its predecessors since the tile was taken --------------
        dec_bar_sync(5 * team + 4 + ((hand - 1) & 1));
        const uint64_t tile_base = s_hand_prefix[(hand - 1) & 1];
        if (tid == 0 && tile > 0)
            st_relaxed_u64(&a.tile_state[tile], (kLbPrefix << kLbFlagShift) | ((tile_base + total) & kLbValueMask));
        for (uint32_t it = tid; it < nitems; it += kDecThreads) b.out_offsets[item0 + it] = tile_base + s_off[it];
        if (tid == 0 && item0 + nitems == b.n) b.out_offsets[b.n] = tile_base + total;
        HB_PHASE_MARK(4);  // wait for the position
        if (staged) {
            const uint64_t room = tile_base < b.out_capacity ? b.out_capacity - tile_base : 0;
            smem_copy_out(s_dense, b.out + tile_base, (uint32_t)min((uint64_t)total, room), tid, kDecThreads);
        } else {
            // ---- write: decode again from global memory, now storing --------------------------------------------------
            for (uint32_t g = warp; g < ngroups;) {
                const uint32_t gslot = g * 32 + lane;
                if (gslot < nitems) {
                    const uint32_t it = s_perm[gslot];
                    const uint64_t off = tile_base + s_off[it];
                    const uint64_t room = off < b.out_capacity ? b.out_capacity - off : 0;
                    const uint64_t in0 = kFramed ? byte0 + (s_start[it] >> 3) - lead : b.in_offsets[item0 + it];
                    const uint64_t len = kFramed ? (uint64_t)s_bytes[it] : b.in_offsets[item0 + it + 1] - in0;
                    if (kFramed && s_cnt[it] == 0) {
                        // nothing to write (empty, malformed or failed literal)
                    } else if (kFramed && (s_flag[it] & 1u)) {
                        for (uint64_t k = 0; k < len && k < room; ++k) b.out[off + k] = b.in[in0 + k];
                    } else {
                        ByteWriter wr;
                        wr.init(b.out + off, room);
                        decode_span_lut2<true>(lut2, b.in + in0, 0, len * 8, len, &wr);
                        wr.finish();
                    }
                }
                uint32_t next = 0;
                if (lane == 0) next = atomicAdd(&s_next, 1u);
                g = __shfl_sync(0xffffffffu, next, 0);
            }
        }
        HB_PHASE_MARK(5);  // image -> global memory
    }
    if (tid == 0) s_hand_tile[hand & 1] = kDecDone;
    dec_bar_arrive(5 * team + 2 + (hand & 1));
}

// ---------------------------------------------------------------------------------------------
// One long stream
//
// Positions are bits in "aligned space": bit 0 is the first bit of the 16-byte aligned block that holds
// the stream's first byte, so chunk k is exactly the aligned words [32k, 32k + 32) and the stream
// occupies [begin_bit, end_bit) = [8 * lead, 8 * (lead + len)).
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kChunkBits = 1024;   // 128 encoded bytes per thread
// Pre-roll: HPACK on Zipf data is in sync after 256 bits for 99.4 % of the starts (SURVEY App. D, longest seen:
// 485), but a tile in which ONE chunk entered wrong pays a whole extra chunk decode with one lane working (the
// others wait at the barrier), and at 256 bits 78 % of the 256-chunk tiles have such a chunk. Measured on the
// 1 GiB stream: 256 bits 2.75 ms, 384 bits 2.47 ms, 512 bits 2.51 ms.
#ifndef HB_PREROLL_BITS
#define HB_PREROLL_BITS 384
#endif
constexpr uint32_t kPrerollBits = HB_PREROLL_BITS;
constexpr int kStreamThreads = 256;
constexpr uint32_t kStreamRowWords = 33;                                      // 32 words + 1 copy of the next row's first
constexpr uint32_t kStreamStageWords = (kStreamThreads + 1) * kStreamRowWords + 1;  // previous chunk + 128 own

// Per-chunk record, one 64-bit word so it is always read and written whole:
//   [15:0]  entry offset  (first code boundary at or after the chunk start, relative to it)
//   [31:16] exit offset   (first code boundary at or after the chunk end, relative to it)
//   [47:32] symbols decoded in the chunk
//   [49:48] termination (kTerm*)
__device__ __forceinline__ uint64_t chunk_pack(uint32_t entry, uint32_t exit, uint32_t nsym, uint32_t term) {
    return (uint64_t)(entry & 0xffffu) | ((uint64_t)(exit & 0xffffu) << 16) | ((uint64_t)(nsym & 0xffffu) << 32) |
           ((uint64_t)(term & 3u) << 48);
}
__device__ __forceinline__ uint32_t chunk_entry(uint64_t w) { return (uint32_t)(w & 0xffffu); }
__device__ __forceinline__ uint32_t chunk_exit(uint64_t w) { return (uint32_t)((w >> 16) & 0xffffu); }
__device__ __forceinline__ uint32_t chunk_nsym(uint64_t w) { return (uint32_t)((w >> 32) & 0xffffu); }
__device__ __forceinline__ uint32_t chunk_term(uint64_t w) { return (uint32_t)((w >> 48) & 3u); }

struct StreamArgs {
    const uint8_t *in_aligned;  // the stream's first byte, rounded down to 16 bytes
    uint64_t begin_bit;         // 8 * lead
    uint64_t end_bit;           // 8 * (lead + len)
    uint64_t num_chunks;
    uint64_t *chunks;           // num_chunks records
    uint64_t *chunk_offsets;    // num_chunks + 1 output offsets (after the scan)
    uint64_t *control;          // [0] = first inconsistent chunk (or ~0), [1] = first terminated chunk (or ~0)
    const uint32_t *lut;
    uint32_t lut_count;
    uint32_t root_bits;
    const uint32_t *gate;       // when set: these kernels only run if *gate != 0 (fallback of the fused kernel)
};
__device__ __forceinline__ bool stream_gate_closed(const StreamArgs &a) { return a.gate != nullptr && *a.gate == 0; }

// (re)decodes one chunk from global memory; used by the rare fix-up paths
__device__ __forceinline__ uint64_t decode_chunk_record(
    const uint32_t *s_lut, const StreamArgs &a, uint64_t k, uint32_t entry) {
    const uint64_t begin = k * kChunkBits;
    const uint64_t stop = min(begin + kChunkBits, a.end_bit);
    const DecodeSpan r =
        decode_span<false, false>(s_lut, a.root_bits, a.in_aligned, begin + entry, stop, a.end_bit >> 3, nullptr);
    const uint32_t exit = r.term == kTermStop ? (uint32_t)(r.pos - stop) : 0u;
    return chunk_pack(entry, exit, (uint32_t)r.nsym, r.term);
}

// Stages chunks [c0 - 1, c0 + kStreamThreads] of the stream as big-endian words in the padded row
// layout and zeroes everything outside the stream. Stage bit 0 is the first bit of chunk c0 - 1.
// in_aligned is 16-byte aligned, so every chunk row is eight 128-bit loads.
__device__ __forceinline__ uint32_t stream_be_word(uint32_t raw, int64_t w, uint64_t end_byte) {
    // big-endian value of aligned word w, with the bytes past the end of the stream cleared
    if (w < 0) return 0;
    const uint64_t first_byte = (uint64_t)w * 4;
    if (first_byte >= end_byte) return 0;
    uint32_t v = __byte_perm(raw, 0, 0x0123);
    if (first_byte + 4 > end_byte) v &= 0xffffffffu << (8 * (first_byte + 4 - end_byte));
    return v;
}

__device__ __forceinline__ void stream_stage(const StreamArgs &a, uint64_t c0, uint32_t *s_in, uint32_t tid) {
    const uint4 *g4 = reinterpret_cast<const uint4 *>(a.in_aligned);
    const uint64_t end_byte = a.end_bit >> 3;
    const uint64_t nquads_valid = (end_byte + 15) >> 4;
    // rows 0..kStreamThreads hold 32 words (8 quads) each; word 32 of a row duplicates word 0 of the next
    constexpr uint32_t kQuads = (kStreamThreads + 1) * 8 + 1;
    if (c0 >= 1 && ((c0 - 1) * 8 + kQuads) * 16 <= end_byte) {
        // interior tile: every staged byte belongs to the stream
        const uint4 *src = g4 + (c0 - 1) * 8;
        for (uint32_t i = tid; i < kQuads; i += kStreamThreads) {
            const uint32_t row = i >> 3, col4 = i & 7;
            const uint4 raw = __ldg(src + i);
            const uint32_t v0 = __byte_perm(raw.x, 0, 0x0123);
            if (row <= kStreamThreads) {
                uint32_t *dst = s_in + row * kStreamRowWords + col4 * 4;
                dst[0] = v0;
                dst[1] = __byte_perm(raw.y, 0, 0x0123);
                dst[2] = __byte_perm(raw.z, 0, 0x0123);
                dst[3] = __byte_perm(raw.w, 0, 0x0123);
            }
            if (col4 == 0 && row > 0) s_in[(row - 1) * kStreamRowWords + 32] = v0;
        }
        return;
    }
    for (uint32_t i = tid; i < kQuads; i += kStreamThreads) {
        const uint32_t row = i >> 3, col4 = i & 7;
        const int64_t q = ((int64_t)c0 - 1 + row) * 8 + col4;  // aligned 16-byte index in the stream
        uint4 raw = make_uint4(0, 0, 0, 0);
        if (q >= 0 && (uint64_t)q < nquads_valid) raw = __ldg(g4 + q);
        const int64_t w = q * 4;
        const uint32_t v0 = stream_be_word(raw.x, w, end_byte);
        if (row <= kStreamThreads) {
            uint32_t *dst = s_in + row * kStreamRowWords + col4 * 4;
            dst[0] = v0;
            dst[1] = stream_be_word(raw.y, w + 1, end_byte);
            dst[2] = stream_be_word(raw.z, w + 2, end_byte);
            dst[3] = stream_be_word(raw.w, w + 3, end_byte);
        }
        if (col4 == 0 && row > 0) s_in[(row - 1) * kStreamRowWords + 32] = v0;
    }
}

// Speculative pass: find an entry point by pre-rolling, then decode the chunk once.
__global__ void __launch_bounds__(kStreamThreads) stream_sync_kernel(StreamArgs a) {
    if (stream_gate_closed(a)) return;
    extern __shared__ uint32_t s_lut[];  // [LUT][stage]
    uint32_t *s_in = s_lut + a.lut_count;
    for (uint32_t i = threadIdx.x; i < a.lut_count; i += kStreamThreads) s_lut[i] = a.lut[i];
    const uint64_t num_tiles = (a.num_chunks + kStreamThreads - 1) / kStreamThreads;
    for (uint64_t t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const uint64_t c0 = t * kStreamThreads;
        __syncthreads();
        stream_stage(a, c0, s_in, threadIdx.x);
        __syncthreads();
        const uint64_t k = c0 + threadIdx.x;
        if (k >= a.num_chunks) continue;
        const uint64_t origin = (c0 - 1) * kChunkBits;  // wraps for c0 == 0; differences below stay exact
        const uint64_t begin = k * kChunkBits;
        const uint64_t stop = min(begin + kChunkBits, a.end_bit);
        const uint32_t s_begin = (uint32_t)(begin - origin), s_stop = (uint32_t)(stop - origin);
        const uint32_t s_end = (uint32_t)min(a.end_bit - origin, (uint64_t)(kStreamThreads + 2) * kChunkBits);
        uint32_t entry;
        if (begin <= a.begin_bit) {
            entry = (uint32_t)(a.begin_bit - begin);  // the stream starts inside this chunk: exact
        } else {
            const uint64_t from = max(begin - kPrerollBits, a.begin_bit);
            const SpanS pre =
                decode_smem<false, true, true>(s_in, s_lut, a.root_bits, (uint32_t)(from - origin), s_begin, s_end, static_cast<WordWriter *>(nullptr));
            entry = pre.pos >= s_begin ? pre.pos - s_begin : 0u;
        }
        const SpanS r = decode_smem<false, true, false>(s_in, s_lut, a.root_bits, s_begin + entry, s_stop, s_end, static_cast<WordWriter *>(nullptr));
        const uint32_t exit = r.term == kTermStop ? r.pos - s_stop : 0u;
        a.chunks[k] = chunk_pack(entry, exit, r.nsym, r.term);
    }
}

// One relaxation round: a chunk whose entry differs from its predecessor's exit is re-decoded from
// there. Records are single words, so updating in place is safe; the fixed point is the true chain.
__global__ void __launch_bounds__(kStreamThreads) stream_fix_kernel(StreamArgs a) {
    if (stream_gate_closed(a)) return;
    extern __shared__ uint32_t s_lut[];
    for (uint32_t i = threadIdx.x; i < a.lut_count; i += kStreamThreads) s_lut[i] = a.lut[i];
    __syncthreads();
    for (uint64_t k = (uint64_t)blockIdx.x * kStreamThreads + threadIdx.x + 1; k < a.num_chunks;
         k += (uint64_t)gridDim.x * kStreamThreads) {
        const uint64_t prev = ld_relaxed_u64(&a.chunks[k - 1]);
        const uint64_t mine = ld_relaxed_u64(&a.chunks[k]);
        if (chunk_term(prev) != kTermStop) continue;  // the stream ended before this chunk
        if (k * kChunkBits <= a.begin_bit) continue;  // the chunk the stream starts in has an exact entry
        if (chunk_entry(mine) != chunk_exit(prev))
            st_relaxed_u64(&a.chunks[k], decode_chunk_record(s_lut, a, k, chunk_exit(prev)));
    }
}

// Finds the first chunk that still disagrees with its predecessor and the first terminated chunk.
__global__ void __launch_bounds__(256) stream_verify_kernel(StreamArgs a) {
    if (stream_gate_closed(a)) return;
    uint64_t bad = ~0ull, term = ~0ull;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < a.num_chunks;
         k += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t mine = a.chunks[k];
        if (chunk_term(mine) != kTermStop && k < term) term = k;
        if (k > 0) {
            const uint64_t prev = a.chunks[k - 1];
            if (chunk_term(prev) == kTermStop && k * kChunkBits > a.begin_bit &&
                chunk_entry(mine) != chunk_exit(prev) && k < bad)
                bad = k;
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, d));
        term = min(term, __shfl_xor_sync(0xffffffffu, term, d));
    }
    if (lane_id() == 0) {
        if (bad != ~0ull) atomicMin(reinterpret_cast<unsigned long long *>(&a.control[0]), (unsigned long long)bad);
        if (term != ~0ull) atomicMin(reinterpret_cast<unsigned long long *>(&a.control[1]), (unsigned long long)term);
    }
}

// Last resort for inputs that do not self-synchronise within a few rounds: one thread walks the chain
// from the first inconsistent chunk. Does nothing when the verify pass found no inconsistency.
__global__ void __launch_bounds__(32) stream_repair_kernel(StreamArgs a) {
    if (stream_gate_closed(a)) return;
    extern __shared__ uint32_t s_lut[];
    if (a.control[0] == ~0ull) return;
    for (uint32_t i = threadIdx.x; i < a.lut_count; i += 32) s_lut[i] = a.lut[i];
    __syncwarp();
    if (threadIdx.x != 0) return;
    uint64_t first_term = a.control[1];
    for (uint64_t k = a.control[0]; k < a.num_chunks; ++k) {
        const uint64_t prev = a.chunks[k - 1];
        if (chunk_term(prev) != kTermStop) break;
        uint64_t mine = a.chunks[k];
        if (chunk_entry(mine) != chunk_exit(prev)) {
            mine = decode_chunk_record(s_lut, a, k, chunk_exit(prev));
            a.chunks[k] = mine;
        }
    }
    // termination may have moved: recompute the first terminated chunk
    first_term = ~0ull;
    for (uint64_t k = 0; k < a.num_chunks; ++k) {
        if (chunk_term(a.chunks[k]) != kTermStop) { first_term = k; break; }
    }
    a.control[1] = first_term;
    a.control[0] = ~0ull;
}

// chunk symbol counts (zero after the first terminated chunk) -> lens array for scan_lens_kernel
__global__ void __launch_bounds__(256) stream_counts_kernel(StreamArgs a, uint64_t *lens) {
    if (stream_gate_closed(a)) return;
    const uint64_t first_term = a.control[1];
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < a.num_chunks;
         k += (uint64_t)gridDim.x * blockDim.x)
        lens[k] = k <= first_term ? chunk_nsym(a.chunks[k]) : 0;
}

// Final pass: every chunk up to the terminating one decodes again, now writing.
__global__ void __launch_bounds__(kStreamThreads) stream_write_kernel(StreamArgs a, BatchView b) {
    if (stream_gate_closed(a)) return;
    extern __shared__ uint32_t s_lut[];  // [LUT][stage]
    uint32_t *s_in = s_lut + a.lut_count;
    for (uint32_t i = threadIdx.x; i < a.lut_count; i += kStreamThreads) s_lut[i] = a.lut[i];
    const uint64_t first_term = a.control[1];
    const uint64_t last = first_term < a.num_chunks ? first_term : a.num_chunks - 1;
    const uint64_t num_tiles = last / kStreamThreads + 1;
    for (uint64_t t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const uint64_t c0 = t * kStreamThreads;
        __syncthreads();
        stream_stage(a, c0, s_in, threadIdx.x);
        __syncthreads();
        const uint64_t k = c0 + threadIdx.x;
        if (k > last) continue;
        const uint64_t origin = (c0 - 1) * kChunkBits;
        const uint64_t rec = a.chunks[k];
        const uint64_t begin = k * kChunkBits;
        const uint64_t stop = min(begin + kChunkBits, a.end_bit);
        const uint32_t s_end = (uint32_t)min(a.end_bit - origin, (uint64_t)(kStreamThreads + 2) * kChunkBits);
        const uint64_t off = a.chunk_offsets[k];
        WordWriter wr;
        wr.init(b.out + off, off < b.out_capacity ? b.out_capacity - off : 0);
        const SpanS r = decode_smem<true, true, false>(
            s_in, s_lut, a.root_bits, (uint32_t)(begin - origin) + chunk_entry(rec), (uint32_t)(stop - origin), s_end, &wr);
        wr.finish();
        if (k == last) {
            // item-level results (n == 1)
            const uint64_t total = off + r.nsym;
            const uint64_t cbits = (uint64_t)r.pos + origin - a.begin_bit;  // stream bits turned into symbols
            b.out_offsets[0] = 0;
            b.out_offsets[1] = total;
            if (b.out_lens) b.out_lens[0] = total;
            if (b.status) b.status[0] = r.term == kTermUnknown ? kStatusUnknownSymbol : kStatusOk;
            if (b.consumed || b.leftover_working_bits || b.leftover_num_bits)
                leftover_state(a.in_aligned + (a.begin_bit >> 3), (a.end_bit - a.begin_bit) >> 3, cbits,
                               r.term == kTermUnknown, b.consumed, b.leftover_working_bits, b.leftover_num_bits);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// One long stream, fused single pass (the normal path; the kernels above remain as the fallback for
// inputs that do not behave, see stream_fused_verify_kernel).
//
// Persistent 256-thread blocks, one chunk per thread, tiles of 256 chunks taken from a ticket:
//   1. stage the tile's chunks (+ the chunk before) in shared memory
//   2. every thread pre-rolls to find its entry point and decodes its chunk ONCE, emitting the symbols
//      byte by byte into a private shared-memory row
//   3. chunks whose entry differs from their predecessor's exit are decoded again from there until the
//      tile is consistent (0.6 % of the chunks on HPACK text). The tile's FIRST chunk is checked against
//      the previous tile: every tile publishes where its last chunk left as soon as it is consistent in
//      itself (never after waiting for another tile: that would chain the waits through the grid), then
//      reads its predecessor's record and, if its first chunk entered elsewhere, decodes again from there.
//      Should that correction ever reach the tile's last chunk (a stream that does not self-synchronise),
//      the published record was wrong and the `fail` flag goes up
//   4. block scan of the symbol counts + decoupled look-back -> output offset of the tile
//   5. rows -> dense image in shared memory (aligned like the global destination) -> 128-bit stores
// The last chunk of the stream absorbs a tail of fewer than 32 bits, so "the stream ended" can only
// be seen by the last chunk. Anything else that stops early (a window that matches no code) raises the
// `fail` flag, and so does a tile whose first chunk did not enter where the previous tile left; the
// fallback kernels then redo the stream (they return at once when the flag is clear).
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kFusedRowSlack = 12;  // bytes: up to 31 / min_len symbols of the absorbed tail, and alignment

struct StreamFusedArgs {
    StreamArgs s;            // num_chunks counts the FUSED chunks: max(1, ceil((end_bit - 31) / kChunkBits))
    BatchView b;
    uint64_t *tile_state;    // look-back descriptors, one per tile
    uint32_t *ticket;
    uint64_t *tile_rec;      // per tile: [15:0] entry of its first chunk, [31:16] exit of its last, [33:32] term of its
                             // last, [63] published
    uint32_t *fail;
    const uint2 *lut2;       // 64-bit entries of the lean step (decode_span_lean)
    uint32_t lut2_count, lut2_trap;
    uint32_t num_tiles;
    uint32_t row_words;      // row stride in words (odd)
};

__device__ __forceinline__ uint64_t fused_chunk_stop(const StreamArgs &a, uint64_t k) {
    return k + 1 == a.num_chunks ? a.end_bit : (k + 1) * kChunkBits;
}

// Shared state of one team of stream_fused_kernel (the two teams of a block share one copy of the decode table,
// see decode_batch_kernel).
struct StreamTeamShared {
    uint16_t entry[kStreamThreads], exit[kStreamThreads];
    uint32_t nsym[kStreamThreads];
    uint8_t term[kStreamThreads];
    uint32_t warp_sum[kStreamThreads / 32];
    uint64_t last_cbits;
    uint32_t tile, first_term, total, last_rel, last_term, flag;
    uint32_t hand_tile[2];     // workers -> scout, by hand-off parity
    uint64_t hand_prefix[2];   // scout -> workers
};
constexpr int kStreamTeams = 2;
constexpr int kStreamTeamThreads = kStreamThreads + 32;  // 8 worker warps + 1 scout warp (see decode_batch_kernel)
// team barriers, 5 per team: workers among themselves 5 t + 1 (plain, and the OR-reduction of a predicate over
// the team); hand-off of a tile to the scout 5 t + 2 + parity; the scout's result 5 t + 4 + parity
__device__ __forceinline__ void stream_team_sync(uint32_t team) { asm volatile("bar.sync %0, %1;" ::"r"(5 * team + 1), "n"(kStreamThreads) : "memory"); }
__device__ __forceinline__ void stream_bar_arrive(uint32_t id) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(kStreamTeamThreads) : "memory"); }
__device__ __forceinline__ void stream_bar_sync(uint32_t id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(kStreamTeamThreads) : "memory"); }
__device__ __forceinline__ bool stream_team_or(uint32_t team, bool pred) {
    uint32_t out;
    asm volatile(
        "{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %1, 0;\n\tbarrier.red.or.pred q, %2, %3, p;\n\tselp.u32 %0, 1, 0, q;\n\t}"
        : "=r"(out)
        : "r"((uint32_t)pred), "r"(5 * team + 1), "n"(kStreamThreads)
        : "memory");
    return out != 0;
}

__global__ void __launch_bounds__(kStreamTeams * kStreamTeamThreads, 1) stream_fused_kernel(StreamFusedArgs f) {
    extern __shared__ __align__(128) uint32_t s_lut[];  // [LUT2][team 0: stage, rows][team 1: stage, rows]
    __shared__ StreamTeamShared s_teams[kStreamTeams];
    const StreamArgs &a = f.s;
    const uint32_t team = threadIdx.x / kStreamTeamThreads, tid = threadIdx.x - team * kStreamTeamThreads;
    StreamTeamShared &sh = s_teams[team];
    uint16_t (&s_entry)[kStreamThreads] = sh.entry, (&s_exit)[kStreamThreads] = sh.exit;
    uint32_t (&s_nsym)[kStreamThreads] = sh.nsym;
    uint8_t (&s_term)[kStreamThreads] = sh.term;
    uint32_t (&s_warp_sum)[kStreamThreads / 32] = sh.warp_sum;
    uint64_t &s_last_cbits = sh.last_cbits;
    uint32_t &s_tile = sh.tile, &s_first_term = sh.first_term, &s_total = sh.total, &s_last_rel = sh.last_rel,
             &s_last_term = sh.last_term;
    const uint32_t lut_pad = 2u * f.lut2_count;
    constexpr uint32_t kStageBytes = (kStreamStageWords * 4 + 15u) & ~15u;
    const uint32_t row_bytes = f.row_words * 4;
    const uint32_t team_bytes = (kStageBytes + kStreamThreads * row_bytes + 16u + 15u) & ~15u;
    uint32_t *s_in = s_lut + lut_pad + team * (team_bytes / 4);
    uint8_t *const s_dense = reinterpret_cast<uint8_t *>(s_in);
    uint8_t *const s_rows = s_dense + kStageBytes;

    const Lut2 lut2 = lut2_load(reinterpret_cast<uint2 *>(s_lut), f.lut2, f.lut2_count, a.root_bits, f.lut2_trap);
    __syncthreads();  // the LUT is in place
    const uint32_t k = tid, lane = lane_id(), warp = tid >> 5;
    // ---- scout: the position of the tile's output (the symbols of all tiles before it), summed next to the
    // tile's own work (see decode_batch_kernel) ---------------------------------------------------------------
    if (warp == kStreamThreads / 32) {
        for (uint32_t h = 0;; ++h) {
            stream_bar_sync(5 * team + 2 + (h & 1));
            const uint32_t t = sh.hand_tile[h & 1];
            if (t == kDecDone) return;
            const uint64_t prefix = lookback_exclusive(f.tile_state, t);
            if (lane == 0) sh.hand_prefix[h & 1] = prefix;
            stream_bar_arrive(5 * team + 4 + (h & 1));
        }
    }
    uint32_t hand = 0;
    const uint32_t row_addr = (uint32_t)__cvta_generic_to_shared(s_rows) + k * row_bytes;

    while (true) {
        stream_team_sync(team);  // previous tile fully done (and the LUT is in place on the first trip)
        if (k == 0) {
            s_tile = atomicAdd(f.ticket, 1u);
            s_first_term = kStreamThreads;
        }
        stream_team_sync(team);
        const uint32_t tile = s_tile;
        if (tile >= f.num_tiles) break;
        if (k == 0) sh.hand_tile[hand & 1] = tile;
        stream_bar_arrive(5 * team + 2 + (hand & 1));  // the scout starts on the tile's position
        ++hand;
        const uint64_t c0 = (uint64_t)tile * kStreamThreads;
        stream_stage(a, c0, s_in, tid);
        stream_team_sync(team);

        // ---- decode my chunk -------------------------------------------------------------------------------------
        const uint64_t chunk = c0 + k;
        const bool valid = chunk < a.num_chunks;
        const uint64_t origin = (c0 - 1) * kChunkBits;  // wraps for c0 == 0; differences below stay exact
        const uint64_t begin = chunk * kChunkBits;
        const uint64_t stop = valid ? fused_chunk_stop(a, chunk) : begin;
        const uint32_t s_begin = (uint32_t)(begin - origin), s_stop = (uint32_t)(stop - origin);
        const uint32_t s_end = (uint32_t)min(a.end_bit - origin, (uint64_t)(kStreamThreads + 2) * kChunkBits);
        const bool exact = begin <= a.begin_bit;  // the stream starts inside this chunk (or after it)
        uint32_t entry = 0, exit = 0, nsym = 0, term = kTermStop;
        uint32_t last_pos = 0;  // stage position after my last symbol (item-level results of the last chunk)
        if (valid) {
            if (exact) {
                entry = (uint32_t)(a.begin_bit - begin);
            } else {
                const uint64_t from = max(begin - kPrerollBits, a.begin_bit);
                const SpanS pre = decode_span_lean<false, true, true>(
                    s_in, lut2, a.root_bits, (uint32_t)(from - origin), s_begin, s_end, 0u);
                entry = pre.pos >= s_begin ? pre.pos - s_begin : 0u;
            }
            const SpanS r = decode_span_lean<true, true, false>(s_in, lut2, a.root_bits, s_begin + entry, s_stop, s_end, row_addr);
            exit = r.term == kTermStop ? r.pos - s_stop : 0u;
            nsym = r.nsym;
            term = r.term;
            last_pos = r.pos;
        }
        // A chunk that did not enter where its predecessor left is decoded again from there. Inside a warp
        // that is settled with shuffles right away (no block barrier, the other warps keep decoding); what
        // is left for the block-wide loop below are the chunks at warp boundaries and the rare cascades.
        while (true) {
            const uint32_t prev_exit = __shfl_up_sync(0xffffffffu, exit, 1);
            const uint32_t prev_term = __shfl_up_sync(0xffffffffu, term, 1);
            const bool redo = valid && lane > 0 && !exact && prev_term == kTermStop && entry != prev_exit;
            if (!__any_sync(0xffffffffu, redo)) break;
            if (redo) {
                const SpanS r = decode_span_lean<true, true, false>(s_in, lut2, a.root_bits, s_begin + prev_exit, s_stop, s_end, row_addr);
                entry = prev_exit;
                exit = r.term == kTermStop ? r.pos - s_stop : 0u;
                nsym = r.nsym;
                term = r.term;
                last_pos = r.pos;
            }
        }
        s_entry[k] = (uint16_t)entry;
        s_exit[k] = (uint16_t)exit;
        s_nsym[k] = nsym;
        s_term[k] = (uint8_t)term;
        stream_team_sync(team);

        // ---- make the tile consistent: in itself, then with the previous tile -----------------------------------
        const uint32_t nvalid = (uint32_t)min((uint64_t)kStreamThreads, a.num_chunks - c0);
        uint32_t prev_exit0 = 0, prev_term0 = kTermEnd;  // thread 0: where the previous tile's last chunk left
        uint64_t published = 0;
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
            while (true) {
                bool redo = false;
                uint32_t want = 0;
                if (valid && !exact) {
                    if (k > 0 && s_term[k - 1] == kTermStop && s_entry[k] != s_exit[k - 1]) {
                        redo = true;
                        want = s_exit[k - 1];
                    } else if (k == 0 && pass == 1 && prev_term0 == kTermStop && s_entry[0] != prev_exit0) {
                        redo = true;
                        want = prev_exit0;
                    }
                }
                if (!stream_team_or(team, redo)) break;
                if (redo) {
                    const SpanS r = decode_span_lean<true, true, false>(s_in, lut2, a.root_bits, s_begin + want, s_stop, s_end, row_addr);
                    s_entry[k] = (uint16_t)want;
                    s_exit[k] = (uint16_t)(r.term == kTermStop ? r.pos - s_stop : 0u);
                    s_nsym[k] = r.nsym;
                    s_term[k] = (uint8_t)r.term;
                    last_pos = r.pos;
                }
                stream_team_sync(team);
            }
            if (k == 0) {
                const uint64_t rec = (1ull << 63) | (uint64_t)s_entry[0] | ((uint64_t)s_exit[nvalid - 1] << 16) |
                                     ((uint64_t)s_term[nvalid - 1] << 32);
                if (pass == 0) {
                    // publish first, then look at the predecessor (which did the same: no chain of waits)
                    published = rec;
                    st_relaxed_u64(&f.tile_rec[tile], rec);
                    if (tile > 0 && !exact) {
                        uint64_t prev;
                        while (((prev = ld_relaxed_u64(&f.tile_rec[tile - 1])) >> 63) == 0) __nanosleep(100);
                        prev_exit0 = (uint32_t)(prev >> 16) & 0xffffu;
                        prev_term0 = (uint32_t)(prev >> 32) & 3u;
                    }
                } else if (rec != published) {
                    st_relaxed_u64(&f.tile_rec[tile], rec);
                    // the correction reached the last chunk: successors may have used the wrong record
                    if ((rec >> 16) != (published >> 16)) atomicExch(f.fail, 1u);
                }
            }
        }
        if (valid && s_term[k] != kTermStop) atomicMin(&s_first_term, k);
        stream_team_sync(team);
        const uint32_t first_term = s_first_term;
        // something stopped before the stream's last chunk: not for this kernel
        if (first_term < kStreamThreads && c0 + first_term + 1 < a.num_chunks && k == 0) atomicExch(f.fail, 1u);

        // ---- offsets: block scan; the tile's count goes out at once ---------------------------------------------
        const uint32_t cnt = (valid && k <= first_term) ? s_nsym[k] : 0u;
        const uint32_t incl = warp_inclusive_scan(cnt);
        if (lane == 31) s_warp_sum[warp] = incl;
        stream_team_sync(team);
        if (warp == 0) {
            const uint32_t w = lane < kStreamThreads / 32 ? s_warp_sum[lane] : 0u;
            const uint32_t wi = warp_inclusive_scan(w);
            if (lane < kStreamThreads / 32) s_warp_sum[lane] = wi - w;
            const uint32_t total = __shfl_sync(0xffffffffu, wi, kStreamThreads / 32 - 1);
            if (lane == 0) {
                lookback_publish_aggregate(f.tile_state, tile, total);
                s_total = total;
            }
        }
        stream_team_sync(team);  // everybody is done with the stage
        const uint32_t off = s_warp_sum[warp] + incl - cnt;
        const uint32_t total = s_total;

        // ---- item-level results (n == 1) come from the stream's last chunk; they go out with its tile ---------
        if (valid && chunk + 1 == a.num_chunks) {
            s_last_rel = off + cnt;
            s_last_cbits = (uint64_t)last_pos + origin - a.begin_bit;  // stream bits turned into symbols
            s_last_term = s_term[k];
        }

        // ---- rows -> dense image in shared memory -> its final place (the scout has the position by now) -----------
        {
            // rows that start before `front` lie where the dense image may grow: they go first (their destination
            // ends inside the stage area); the image (<= 256 rows) ends before row offset `front` + stage
            const uint32_t front = kStageBytes - row_bytes - 32;
            const uint32_t row_off = k * row_bytes;
#pragma unroll 1
            for (int phase = 0; phase < 2; ++phase) {
#ifndef HB_ABL_NO_COPY
                if ((row_off < front) == (phase == 0)) smem_copy_row(s_rows + row_off, s_dense + off, cnt);
#endif
                stream_team_sync(team);
            }
        }
        stream_bar_sync(5 * team + 4 + ((hand - 1) & 1));
        const uint64_t tile_base = sh.hand_prefix[(hand - 1) & 1];
        if (k == 0 && tile > 0)
            st_relaxed_u64(&f.tile_state[tile], (kLbPrefix << kLbFlagShift) | ((tile_base + total) & kLbValueMask));
        if (tile == f.num_tiles - 1 && k == 0) {
            const BatchView &b = f.b;
            const uint64_t nsym_all = tile_base + s_last_rel;
            b.out_offsets[0] = 0;
            b.out_offsets[1] = nsym_all;
            if (b.out_lens) b.out_lens[0] = nsym_all;
            if (b.status) b.status[0] = s_last_term == kTermUnknown ? kStatusUnknownSymbol : kStatusOk;
            if (b.consumed || b.leftover_working_bits || b.leftover_num_bits)
                leftover_state(a.in_aligned + (a.begin_bit >> 3), (a.end_bit - a.begin_bit) >> 3, s_last_cbits,
                               s_last_term == kTermUnknown, b.consumed, b.leftover_working_bits, b.leftover_num_bits);
        }
        {
            const uint64_t room = tile_base < f.b.out_capacity ? f.b.out_capacity - tile_base : 0;
            smem_copy_out(s_dense, f.b.out + tile_base, (uint32_t)min((uint64_t)total, room), k, kStreamThreads);
        }
    }
    if (k == 0) sh.hand_tile[hand & 1] = kDecDone;
    stream_bar_arrive(5 * team + 2 + (hand & 1));
}

// Every tile's first chunk must have entered exactly where the previous tile's last chunk left.
__global__ void __launch_bounds__(256) stream_fused_verify_kernel(StreamFusedArgs f) {
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x + 1; t < f.num_tiles; t += gridDim.x * blockDim.x) {
        const uint64_t prev = f.tile_rec[t - 1], mine = f.tile_rec[t];
        const uint32_t prev_exit = (uint32_t)(prev >> 16) & 0xffffu, prev_term = (uint32_t)(prev >> 32) & 3u;
        if (prev_term != kTermStop || (uint32_t)(mine & 0xffffu) != prev_exit) atomicExch(f.fail, 1u);
    }
}

}  // namespace hb
