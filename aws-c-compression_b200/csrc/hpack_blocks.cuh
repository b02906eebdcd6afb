// HPACK header blocks (RFC 7541 section 6 representations, Appendix A static table) around the string-literal
// layer of hpack_literals.cuh.
//
//     indexed              1xxxxxxx   index, 7-bit prefix (0 is an error)
//     literal, incremental 01xxxxxx   name index, 6-bit prefix (0: a name literal follows), value literal
//     literal, without     0000xxxx   name index, 4-bit prefix, ...
//     literal, never       0001xxxx   name index, 4-bit prefix, ...
//     size update          001xxxxx   new maximum size, 5-bit prefix (only before the first field of a block)
//
// Decode: one thread walks one block (the representations are sequential: where one starts is known only when the
// previous one was read), twice: once to count fields, literals and literal octets, once to write the field records
// and the literal spans. The literals are gathered into a packed batch and decoded by the literal path
// (hpack_decode_on_device, either route); then a per-block pass picks the final status and per-field passes write
// the records and the strings, each from the static table below or from the decoded literals.
// Encode: one thread per field picks its representation (the caller's record, or a match against the static table);
// every name and value is framed by the literal path; for records, one thread per block applies the block rules;
// a warp per 32 fields writes the prefix integers and copies the framed literals the representation uses.
#pragma once

#include "hpack_literals.cuh"

namespace hb {

enum : uint8_t { kFieldIndexed = 0, kFieldIncremental = 1, kFieldWithout = 2, kFieldNever = 3, kFieldSizeUpdate = 4 };
constexpr uint64_t kNoLiteral = ~0ull;
constexpr uint32_t kStaticEntries = 61;

// RFC 7541 Appendix A: entry i (1-based) has its name at [kStaticOff[2i-2], kStaticOff[2i-1]) and its value at
// [kStaticOff[2i-1], kStaticOff[2i]) of kStaticBlob.
__device__ const uint8_t kStaticBlob[] =
    ":authority"
    ":method" "GET" ":method" "POST" ":path" "/" ":path" "/index.html" ":scheme" "http" ":scheme" "https"
    ":status" "200" ":status" "204" ":status" "206" ":status" "304" ":status" "400" ":status" "404" ":status" "500"
    "accept-charset" "accept-encoding" "gzip, deflate" "accept-language" "accept-ranges" "accept"
    "access-control-allow-origin" "age" "allow" "authorization" "cache-control" "content-disposition"
    "content-encoding" "content-language" "content-length" "content-location" "content-range" "content-type"
    "cookie" "date" "etag" "expect" "expires" "from" "host" "if-match" "if-modified-since" "if-none-match"
    "if-range" "if-unmodified-since" "last-modified" "link" "location" "max-forwards" "proxy-authenticate"
    "proxy-authorization" "range" "referer" "refresh" "retry-after" "server" "set-cookie"
    "strict-transport-security" "transfer-encoding" "user-agent" "vary" "via" "www-authenticate";
static_assert(sizeof(kStaticBlob) == 684 + 1, "Appendix A holds 684 octets of names and values");
__device__ const uint16_t kStaticOff[2 * kStaticEntries + 1] = {
    0,   10,  10,  17,  20,  27,  31,  36,  37,  42,  53,  60,  64,  71,  76,  83,  86,  93,  96,  103, 106,
    113, 116, 123, 126, 133, 136, 143, 146, 160, 160, 175, 188, 203, 203, 216, 216, 222, 222, 249, 249, 252,
    252, 257, 257, 270, 270, 283, 283, 302, 302, 318, 318, 334, 334, 348, 348, 364, 364, 377, 377, 389, 389,
    395, 395, 399, 399, 403, 403, 409, 409, 416, 416, 420, 420, 424, 424, 432, 432, 449, 449, 462, 462, 470,
    470, 489, 489, 502, 502, 506, 506, 514, 514, 526, 526, 544, 544, 563, 563, 568, 568, 575, 575, 582, 582,
    593, 593, 599, 599, 609, 609, 634, 634, 651, 651, 661, 661, 665, 665, 668, 668, 684, 684};

// ---- integers (RFC 7541 5.1) ------------------------------------------------------------------------------------
// Reads the integer whose first octet is p[pos] (pos < end); same limit as hpack_parse_literal: at most 9
// continuation octets are taken, a tenth is INVALID_ARGUMENT.
__device__ __forceinline__ int32_t hpack_read_int(const uint8_t *p, uint64_t end, uint64_t &pos, uint32_t prefix_bits,
                                                  uint64_t &value) {
    const uint32_t limit = (1u << prefix_bits) - 1;
    value = p[pos++] & limit;
    if (value < limit) return kStatusOk;
    uint32_t shift = 0;
    for (;;) {
        if (pos >= end) return kStatusShortBuffer;
        const uint8_t b = p[pos++];
        if (shift > 56) return kStatusInvalidArgument;
        value += (uint64_t)(b & 127) << shift;
        shift += 7;
        if (!(b & 128)) return kStatusOk;
    }
}

__device__ __forceinline__ uint32_t hpack_int_bytes(uint64_t v, uint32_t prefix_bits) {
    const uint32_t limit = (1u << prefix_bits) - 1;
    if (v < limit) return 1;
    uint32_t nb = 2;
    for (uint64_t rem = v - limit; rem >= 128; rem >>= 7) ++nb;
    return nb;
}

// Writes the integer at out[pos ..) with `flags` in the first octet's high bits; nothing at or after `cap`.
__device__ __forceinline__ void hpack_put_int(uint8_t *out, uint64_t pos, uint64_t cap, uint64_t v, uint32_t prefix_bits,
                                              uint8_t flags) {
    const uint32_t limit = (1u << prefix_bits) - 1;
    if (v < limit) {
        if (pos < cap) out[pos] = flags | (uint8_t)v;
        return;
    }
    if (pos < cap) out[pos] = flags | (uint8_t)limit;
    ++pos;
    for (v -= limit; v >= 128; v >>= 7, ++pos)
        if (pos < cap) out[pos] = (uint8_t)(v & 127) | 0x80;
    if (pos < cap) out[pos] = (uint8_t)v;
}

// ---- decode: the structural walk -----------------------------------------------------------------------------
struct BlockField {
    uint8_t kind;
    bool complete;             // false: the field failed after its name literal; only that literal is reported
    bool name_lit, value_lit;  // which literal spans below were read in full
    uint64_t index;
    // literal spans (prefix and payload), relative to the block (separate fields, not an array: a dynamically indexed
    // array would live in local memory)
    uint64_t name_begin, name_end, value_begin, value_end;
};

// One string literal at p[pos ..): its span, or the error a decoder meets inside it.
__device__ __forceinline__ int32_t hpack_skip_literal(const uint8_t *p, uint64_t end, uint64_t &pos, uint64_t &begin,
                                                      uint64_t &stop) {
    begin = pos;
    if (pos >= end) return kStatusShortBuffer;
    uint64_t len;
    const int32_t st = hpack_read_int(p, end, pos, 7, len);
    if (st != kStatusOk) return st;
    if (len > end - pos) return kStatusShortBuffer;
    pos += len;
    stop = pos;
    return kStatusOk;
}

// Walks one block front to back and calls visit(field) for every representation read in full. Returns the first
// structural error (the walk stops there) or kStatusOk. Huffman payloads are not looked at here. When a field fails
// after its name literal was read in full, that literal lies before the error and a front-to-back decoder decodes it
// first, so its own errors must win: it is visited too, as an incomplete field (a literal that belongs to no field).
template <typename Visit>
__device__ __forceinline__ int32_t hpack_walk_block(const uint8_t *p, uint64_t size, Visit &&visit) {
    uint64_t pos = 0;
    bool seen_field = false;
    while (pos < size) {
        const uint8_t b0 = p[pos];
        BlockField f;
        f.complete = true;
        f.name_lit = f.value_lit = false;
        int32_t st;
        if (b0 & 0x80) {
            f.kind = kFieldIndexed;
            st = hpack_read_int(p, size, pos, 7, f.index);
            if (st == kStatusOk && f.index == 0) st = kStatusInvalidArgument;
        } else if ((b0 & 0xe0) == 0x20) {
            f.kind = kFieldSizeUpdate;  // (an update after a field is refused at its first octet)
            st = seen_field ? kStatusInvalidArgument : hpack_read_int(p, size, pos, 5, f.index);
        } else {
            f.kind = (b0 & 0x40) ? kFieldIncremental : ((b0 & 0x10) ? kFieldNever : kFieldWithout);
            st = hpack_read_int(p, size, pos, (b0 & 0x40) ? 6 : 4, f.index);
            if (st == kStatusOk && f.index == 0) {
                st = hpack_skip_literal(p, size, pos, f.name_begin, f.name_end);
                f.name_lit = st == kStatusOk;
            }
            if (st == kStatusOk) {
                st = hpack_skip_literal(p, size, pos, f.value_begin, f.value_end);
                f.value_lit = st == kStatusOk;
            }
        }
        if (st != kStatusOk) {
            if (f.name_lit) {
                f.complete = false;
                visit(f);
            }
            return st;
        }
        seen_field |= f.kind != kFieldSizeUpdate;
        visit(f);
    }
    return kStatusOk;
}

// Pass 1, thread per block: fields and literals read before the first structural error (a failing field's name
// literal included), their literal octets, and that error.
__global__ void hpack_block_scan_kernel(uint64_t n, const uint8_t *in, const uint64_t *in_offsets, uint64_t *num_fields,
                                        uint64_t *num_lits, uint64_t *lit_bytes, int32_t *struct_status) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t a = in_offsets[b];
    uint64_t nf = 0, nl = 0, nbytes = 0;
    struct_status[b] = hpack_walk_block(in + a, in_offsets[b + 1] - a, [&](const BlockField &f) {
        nf += f.complete;
        nl += f.name_lit + f.value_lit;
        if (f.name_lit) nbytes += f.name_end - f.name_begin;
        if (f.value_lit) nbytes += f.value_end - f.value_begin;
    });
    num_fields[b] = nf;
    num_lits[b] = nl;
    lit_bytes[b] = nbytes;
}

// Pass 2, thread per block, the same walk: field records (kind, index, block, the literal ids of name and value)
// in parsed order from field_base[b], and literal spans (source offset into `in`, offset in the packed literal
// batch) from lit_base[b] / lit_byte_base[b]. An incomplete field gets its literal span and no record.
__global__ void hpack_block_split_kernel(
    uint64_t n, const uint8_t *in, const uint64_t *in_offsets, const uint64_t *field_base, const uint64_t *lit_base,
    const uint64_t *lit_byte_base, uint8_t *f_kind, uint64_t *f_index, uint32_t *f_block, uint64_t *f_lits,
    uint64_t *lit_src, uint64_t *lit_offsets) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t a = in_offsets[b];
    uint64_t f = field_base[b], l = lit_base[b], o = lit_byte_base[b];
    hpack_walk_block(in + a, in_offsets[b + 1] - a, [&](const BlockField &fd) {
        uint64_t name = kNoLiteral, value = kNoLiteral;
        if (fd.name_lit) {
            name = l;
            lit_src[l] = a + fd.name_begin;
            lit_offsets[l++] = o;
            o += fd.name_end - fd.name_begin;
        }
        if (fd.value_lit) {
            value = l;
            lit_src[l] = a + fd.value_begin;
            lit_offsets[l++] = o;
            o += fd.value_end - fd.value_begin;
        }
        if (!fd.complete) return;
        f_kind[f] = fd.kind;
        f_index[f] = fd.index;
        f_block[f] = (uint32_t)b;
        f_lits[2 * f] = name;
        f_lits[2 * f + 1] = value;
        ++f;
    });
    if (b == n - 1) lit_offsets[l] = o;
}

// The literals, packed (lit_offsets) for the literal decoder. 32 literals per warp (warp_run_jobs).
__global__ void __launch_bounds__(256) hpack_lit_gather_kernel(
    uint64_t num_lits, const uint8_t *in, const uint64_t *lit_src, const uint64_t *lit_offsets, uint8_t *dst) {
    __shared__ MoveJob s_jobs[8][32];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint64_t l = ((uint64_t)blockIdx.x * 8 + warp) * 32 + lane;
    MoveJob job = {nullptr, nullptr, 0};
    if (l < num_lits) {
        job.src = in + lit_src[l];
        job.dst = dst + lit_offsets[l];
        job.len = lit_offsets[l + 1] - lit_offsets[l];
    }
    warp_run_jobs(s_jobs, job, warp, lane);
}

// Thread per block: the final status and the number of fields the block yields. The walk stopped at the structural
// error, and every literal it reported (the name literal of the field that failed included) ends before that error:
// the first failing literal, if any, is the first error in byte order.
__global__ void hpack_block_finish_kernel(
    uint64_t n, const uint64_t *lit_base, const int32_t *lit_status, const int32_t *struct_status,
    const uint64_t *num_fields, int32_t *status, uint64_t *out_fields) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    int32_t st = kStatusOk;
    for (uint64_t l = lit_base[b]; l < lit_base[b + 1] && st == kStatusOk; ++l) st = lit_status[l];
    if (st == kStatusOk) st = struct_status[b];
    status[b] = st;
    out_fields[b] = st == kStatusOk ? num_fields[b] : 0;
}

// Where one string of a parsed field comes from: its decoded literal, the static table, or nowhere (a dynamic
// reference or a size update: empty).
__device__ __forceinline__ void hpack_field_string(
    uint8_t kind, uint64_t index, uint64_t lit, uint32_t which, const uint8_t *dec, const uint64_t *dec_offsets,
    const uint8_t *&src, uint64_t &len) {
    src = nullptr;
    len = 0;
    if (lit != kNoLiteral) {
        src = dec + dec_offsets[lit];
        len = dec_offsets[lit + 1] - dec_offsets[lit];
    } else if (kind != kFieldSizeUpdate && index >= 1 && index <= kStaticEntries && (which == 0 || kind == kFieldIndexed)) {
        const uint32_t e = 2 * (uint32_t)(index - 1) + which;
        src = kStaticBlob + kStaticOff[e];
        len = kStaticOff[e + 1] - kStaticOff[e];
    }
}

// The output slot of parsed field f, or ~0 when its block failed or it lies beyond field_capacity.
__device__ __forceinline__ uint64_t hpack_out_field(
    uint64_t f, const uint32_t *f_block, const uint64_t *field_base, const int32_t *status, const uint64_t *field_offsets,
    uint64_t field_capacity) {
    const uint32_t b = f_block[f];
    if (status[b] != kStatusOk) return ~0ull;
    const uint64_t o = field_offsets[b] + (f - field_base[b]);
    return o < field_capacity ? o : ~0ull;
}

// The string source of HPACK fields for hpack_field_records_kernel and hpack_compose_kernel (qpack_sections.cuh and
// qpack_instructions.cuh have QPACK's).
struct HpackFieldStrings {
    __device__ static void get(uint8_t kind, uint64_t index, uint64_t lit, uint32_t which, const uint8_t *dec,
                               const uint64_t *dec_offsets, const uint8_t *&src, uint64_t &len) {
        hpack_field_string(kind, index, lit, which, dec, dec_offsets, src, len);
    }
};

// Thread per parsed field: the record and the lengths of its two strings (Strings::get says where a string of a
// parsed field comes from).
template <typename Strings>
__global__ void hpack_field_records_kernel(
    uint64_t num_parsed, const uint8_t *f_kind, const uint64_t *f_index, const uint32_t *f_block, const uint64_t *f_lits,
    const uint64_t *field_base, const int32_t *status, const uint64_t *field_offsets, uint64_t field_capacity,
    const uint8_t *dec, const uint64_t *dec_offsets, uint8_t *out_kind, uint64_t *out_index, uint64_t *str_lens) {
    const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= num_parsed) return;
    const uint64_t o = hpack_out_field(f, f_block, field_base, status, field_offsets, field_capacity);
    if (o == ~0ull) return;
    const uint8_t kind = f_kind[f];
    const uint64_t index = f_index[f];
    out_kind[o] = kind;
    out_index[o] = index;
    for (uint32_t w = 0; w < 2; ++w) {
        const uint8_t *src;
        uint64_t len;
        Strings::get(kind, index, f_lits[2 * f + w], w, dec, dec_offsets, src, len);
        str_lens[2 * o + w] = len;
    }
}

// The strings: item i is string i & 1 (name, value) of parsed field i >> 1. 32 strings per warp. Strings::get says
// where a string of a parsed field comes from.
template <typename Strings>
__global__ void __launch_bounds__(256) hpack_compose_kernel(
    uint64_t num_parsed, const uint8_t *f_kind, const uint64_t *f_index, const uint32_t *f_block, const uint64_t *f_lits,
    const uint64_t *field_base, const int32_t *status, const uint64_t *field_offsets, uint64_t field_capacity,
    const uint8_t *dec, const uint64_t *dec_offsets, uint8_t *strings, uint64_t strings_capacity,
    const uint64_t *string_offsets) {
    __shared__ MoveJob s_jobs[8][32];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint64_t i = ((uint64_t)blockIdx.x * 8 + warp) * 32 + lane;
    MoveJob job = {nullptr, nullptr, 0};
    if (i < 2 * num_parsed) {
        const uint64_t f = i >> 1;
        const uint32_t w = (uint32_t)(i & 1);
        const uint64_t o = hpack_out_field(f, f_block, field_base, status, field_offsets, field_capacity);
        if (o != ~0ull) {
            const uint8_t *src;
            uint64_t len;
            Strings::get(f_kind[f], f_index[f], f_lits[2 * f + w], w, dec, dec_offsets, src, len);
            const uint64_t o0 = string_offsets[2 * o + w];
            const uint64_t room = o0 < strings_capacity ? strings_capacity - o0 : 0;
            job.src = src;
            job.dst = strings + o0;
            job.len = min(len, room);
        }
    }
    warp_run_jobs(s_jobs, job, warp, lane);
}

// ---- encode ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool hpack_bytes_equal(const uint8_t *a, const uint8_t *b, uint64_t len) {
    for (uint64_t k = 0; k < len; ++k)
        if (a[k] != b[k]) return false;
    return true;
}

// Plan byte of a field: representation in bits 0..2, "name literal" in bit 3, "value literal" in bit 4, "emit
// nothing" in bit 5 (the field is invalid, or its block is); the index or size in plan_index.
enum : uint8_t { kPlanNameLit = 8, kPlanValueLit = 16, kPlanSkip = 32 };
// A record's kind on the encode side: the five representations, or the stateless rules (kFieldAuto).
constexpr uint8_t kFieldAuto = 5;

// Prefix bits and first-octet flags of each representation (RFC 7541 6.1 - 6.3).
__device__ __forceinline__ uint32_t hpack_prefix_bits(uint32_t kind) { return 0x54467u >> (4 * kind) & 15; }  // 7 6 4 4 5
__device__ __forceinline__ uint8_t hpack_prefix_flags(uint32_t kind) {
    return (uint8_t)(0x2010004080ull >> (8 * kind));  // 0x80 0x40 0x00 0x10 0x20
}

// Thread per field: representation and the field's size on the wire from the framed literals (framed_offsets: name
// of field f is framed item 2f, its value 2f + 1). field_kind == NULL: every field is kFieldAuto (the rules of
// aws_hpack_header_block_encode_batch); else the caller's kind and field_index[f] are used as given. A field whose
// kind is unknown, an INDEXED index 0, or an integer that hpack_read_int refuses (more than 9 continuation octets)
// gets kPlanSkip and length 0.
__global__ void hpack_field_plan_kernel(
    uint64_t num_fields, const uint8_t *strings, const uint64_t *string_offsets, const uint8_t *never_indexed,
    const uint8_t *field_kind, const uint64_t *field_index, const uint64_t *framed_offsets, uint8_t *plan,
    uint64_t *plan_index, uint64_t *field_lens) {
    const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= num_fields) return;
    const uint8_t kind = field_kind ? field_kind[f] : kFieldAuto;
    uint8_t p;
    uint64_t index;
    if (kind == kFieldAuto) {
        const uint64_t n0 = string_offsets[2 * f], v0 = string_offsets[2 * f + 1], v1 = string_offsets[2 * f + 2];
        const uint8_t *name = strings + n0, *value = strings + v0;
        const uint64_t name_len = v0 - n0, value_len = v1 - v0;
        uint32_t name_match = 0, exact = 0;
        for (uint32_t e = 1; e <= kStaticEntries && !exact; ++e) {
            const uint32_t s0 = kStaticOff[2 * e - 2], s1 = kStaticOff[2 * e - 1], s2 = kStaticOff[2 * e];
            if (s1 - s0 != name_len || !hpack_bytes_equal(name, kStaticBlob + s0, name_len)) continue;
            if (!name_match) name_match = e;
            if (s2 - s1 == value_len && hpack_bytes_equal(value, kStaticBlob + s1, value_len)) exact = e;
        }
        const bool never = never_indexed && never_indexed[f];
        if (!never && exact) {
            p = kFieldIndexed;
            index = exact;
        } else {
            p = (never ? kFieldNever : kFieldWithout) | kPlanValueLit | (name_match ? 0 : kPlanNameLit);
            index = name_match;
        }
    } else if (kind < kFieldAuto) {
        index = field_index[f];
        p = kind;
        if (kind != kFieldIndexed && kind != kFieldSizeUpdate) p |= kPlanValueLit | (index ? 0 : kPlanNameLit);
        if (kind == kFieldIndexed && index == 0) p |= kPlanSkip;
    } else {
        p = kPlanSkip;
        index = 0;
    }
    uint64_t len = 0;
    if (!(p & kPlanSkip)) {
        len = hpack_int_bytes(index, hpack_prefix_bits(p & 7));
        if (len > 10) p |= kPlanSkip;
        if (p & kPlanNameLit) len += framed_offsets[2 * f + 1] - framed_offsets[2 * f];
        if (p & kPlanValueLit) len += framed_offsets[2 * f + 2] - framed_offsets[2 * f + 1];
    }
    plan[f] = p;
    plan_index[f] = index;
    field_lens[f] = p & kPlanSkip ? 0 : len;
}

// Thread per block, after the plan and before the scan of field lengths (records only): a block is invalid when a
// field of it is marked kPlanSkip, or when a size update follows a field that is not one (the decoder's rule). An
// invalid block gets INVALID_ARGUMENT and every field of it kPlanSkip and length 0: it encodes to zero octets.
__global__ void hpack_block_check_kernel(uint64_t n, const uint64_t *field_offsets, uint8_t *plan, uint64_t *field_lens,
                                         int32_t *status) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t f0 = field_offsets[b], f1 = field_offsets[b + 1];
    bool ok = true, seen_field = false;
    for (uint64_t f = f0; f < f1 && ok; ++f) {
        const uint8_t p = plan[f], kind = p & 7;
        ok = !(p & kPlanSkip) && !(kind == kFieldSizeUpdate && seen_field);
        seen_field |= kind != kFieldSizeUpdate;
    }
    if (status) status[b] = ok ? kStatusOk : kStatusInvalidArgument;
    if (ok) return;
    for (uint64_t f = f0; f < f1; ++f) {
        plan[f] |= kPlanSkip;
        field_lens[f] = 0;
    }
}

// out_offsets[b] = the wire position of list b's first field.
__global__ void hpack_block_offsets_kernel(uint64_t n, const uint64_t *field_offsets, const uint64_t *field_pos,
                                           uint64_t *out_offsets) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b <= n) out_offsets[b] = field_pos[field_offsets[b]];
}

// A warp takes 32 fields: every lane writes its field's prefix integer, then the warp copies the 32 name literals
// and the 32 value literals (those the plan uses). Fields marked kPlanSkip write nothing. Never writes at or after
// out + out_capacity.
__global__ void __launch_bounds__(256) hpack_field_emit_kernel(
    uint64_t num_fields, const uint8_t *plan, const uint64_t *plan_index, const uint8_t *framed,
    const uint64_t *framed_offsets, const uint64_t *field_pos, uint8_t *out, uint64_t out_capacity) {
    __shared__ MoveJob s_jobs[8][32];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint64_t f = ((uint64_t)blockIdx.x * 8 + warp) * 32 + lane;
    MoveJob name = {nullptr, nullptr, 0}, value = {nullptr, nullptr, 0};
    if (f < num_fields && !(plan[f] & kPlanSkip)) {
        const uint8_t p = plan[f], kind = p & 7;
        const uint64_t index = plan_index[f];
        uint64_t pos = field_pos[f];
        const uint32_t prefix_bits = hpack_prefix_bits(kind);
        hpack_put_int(out, pos, out_capacity, index, prefix_bits, hpack_prefix_flags(kind));
        pos += hpack_int_bytes(index, prefix_bits);
        for (uint32_t w = 0; w < 2; ++w) {
            if (!(p & (w ? kPlanValueLit : kPlanNameLit))) continue;
            const uint64_t a = framed_offsets[2 * f + w], len = framed_offsets[2 * f + w + 1] - a;
            MoveJob &j = w ? value : name;
            j.src = framed + a;
            j.dst = out + pos;
            j.len = pos < out_capacity ? min(len, out_capacity - pos) : 0;
            pos += len;
        }
    }
    warp_run_jobs(s_jobs, name, warp, lane);
    __syncwarp();
    warp_run_jobs(s_jobs, value, warp, lane);
}

}  // namespace hb
