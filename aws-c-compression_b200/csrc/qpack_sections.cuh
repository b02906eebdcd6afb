// QPACK field sections (RFC 9204 section 4.5 field lines, Appendix A static table) around the string-literal layer
// of hpack_literals.cuh, with the integers and the pipeline of hpack_blocks.cuh.
//
//     section prefix       Encoded Required Insert Count (8-bit prefix), then S and Delta Base (7-bit prefix)
//     indexed              1Txxxxxx   index, 6-bit prefix (T: static, else relative)
//     indexed, post-base   0001xxxx   post-base index, 4-bit prefix
//     name reference       01NTxxxx   name index, 4-bit prefix (T: static, else relative), value literal
//     name ref, post-base  0000Nxxx   post-base name index, 3-bit prefix, value literal
//     literal name         001NHxxx   name length, 3-bit prefix, name payload (H: Huffman), value literal
//
// Decode: the walk of hpack_blocks.cuh (thread per section, twice: counts, then records and literal spans). The
// gather writes every literal into the packed batch re-framed as an RFC 7541 5.2 literal (H in bit 7, a 7-bit-prefix
// length, the payload), so the HPACK literal decoder (hpack_decode_on_device, either route) decodes QPACK literals
// unchanged: value literals already have that framing, name literals change only their first octets.
// Encode: names and values are framed by the literal path; one thread per field picks the line (the caller's record,
// or a match against the static table); one thread per section checks the records and sizes the section (prefix
// included: a section without fields is still two octets or more); one thread per section writes its prefix and
// places its fields; a warp per 32 fields writes their integers and copies the literals, a name literal re-framed
// into the 3-bit form.
#pragma once

#include "hpack_blocks.cuh"

namespace hb {

enum : uint8_t {
    kQIndexedStatic = 0,
    kQIndexedDynamic = 1,
    kQIndexedPostBase = 2,
    kQNameRefStatic = 3,
    kQNameRefDynamic = 4,
    kQNameRefPostBase = 5,
    kQLiteralName = 6,
    kQAuto = 7,  // encode records only: the stateless rules choose
};
constexpr uint32_t kQpackStaticEntries = 99;
constexpr uint8_t kQNeverBit = 8;  // parsed field kinds: the N bit beside the kind

// RFC 9204 Appendix A: entry i (0-based) has its name at [kQpackStaticOff[2i], kQpackStaticOff[2i+1]) and its value
// at [kQpackStaticOff[2i+1], kQpackStaticOff[2i+2]) of kQpackStaticBlob.
__device__ const uint8_t kQpackStaticBlob[] =
    ":authority" ":path" "/" "age" "0" "content-disposition" "content-length" "0" "cookie" "date" "etag"
    "if-modified-since" "if-none-match" "last-modified" "link" "location" "referer" "set-cookie" ":method" "CONNECT"
    ":method" "DELETE" ":method" "GET" ":method" "HEAD" ":method" "OPTIONS" ":method" "POST" ":method" "PUT" ":scheme"
    "http" ":scheme" "https" ":status" "103" ":status" "200" ":status" "304" ":status" "404" ":status" "503" "accept"
    "*/*" "accept" "application/dns-message" "accept-encoding" "gzip, deflate, br" "accept-ranges" "bytes"
    "access-control-allow-headers" "cache-control" "access-control-allow-headers" "content-type"
    "access-control-allow-origin" "*" "cache-control" "max-age=0" "cache-control" "max-age=2592000" "cache-control"
    "max-age=604800" "cache-control" "no-cache" "cache-control" "no-store" "cache-control" "public, max-age=31536000"
    "content-encoding" "br" "content-encoding" "gzip" "content-type" "application/dns-message" "content-type"
    "application/javascript" "content-type" "application/json" "content-type" "application/x-www-form-urlencoded"
    "content-type" "image/gif" "content-type" "image/jpeg" "content-type" "image/png" "content-type" "text/css"
    "content-type" "text/html; charset=utf-8" "content-type" "text/plain" "content-type" "text/plain;charset=utf-8"
    "range" "bytes=0-" "strict-transport-security" "max-age=31536000" "strict-transport-security"
    "max-age=31536000; includesubdomains" "strict-transport-security" "max-age=31536000; includesubdomains; preload"
    "vary" "accept-encoding" "vary" "origin" "x-content-type-options" "nosniff" "x-xss-protection" "1; mode=block"
    ":status" "100" ":status" "204" ":status" "206" ":status" "302" ":status" "400" ":status" "403" ":status" "421"
    ":status" "425" ":status" "500" "accept-language" "access-control-allow-credentials" "FALSE"
    "access-control-allow-credentials" "TRUE" "access-control-allow-headers" "*" "access-control-allow-methods" "get"
    "access-control-allow-methods" "get, post, options" "access-control-allow-methods" "options"
    "access-control-expose-headers" "content-length" "access-control-request-headers" "content-type"
    "access-control-request-method" "get" "access-control-request-method" "post" "alt-svc" "clear" "authorization"
    "content-security-policy" "script-src 'none'; object-src 'none'; base-uri 'none'" "early-data" "1" "expect-ct"
    "forwarded" "if-range" "origin" "purpose" "prefetch" "server" "timing-allow-origin" "*"
    "upgrade-insecure-requests" "1" "user-agent" "x-forwarded-for" "x-frame-options" "deny" "x-frame-options"
    "sameorigin";
static_assert(sizeof(kQpackStaticBlob) == 2026 + 1, "RFC 9204 Appendix A holds 2026 octets of names and values");
__device__ const uint16_t kQpackStaticOff[2 * kQpackStaticEntries + 1] = {
    0, 10, 10, 15, 16, 19, 20, 39, 39, 53, 54, 60, 60, 64, 64, 68, 68, 85, 85, 98, 98, 111, 111, 115, 115, 123, 123,
    130, 130, 140, 140, 147, 154, 161, 167, 174, 177, 184, 188, 195, 202, 209, 213, 220, 223, 230, 234, 241, 246, 253,
    256, 263, 266, 273, 276, 283, 286, 293, 296, 302, 305, 311, 334, 349, 366, 379, 384, 412, 425, 453, 465, 492, 493,
    506, 515, 528, 543, 556, 570, 583, 591, 604, 612, 625, 649, 665, 667, 683, 687, 699, 722, 734, 756, 768, 784, 796,
    829, 841, 850, 862, 872, 884, 893, 905, 913, 925, 949, 961, 971, 983, 1007, 1012, 1020, 1045, 1061, 1086, 1121,
    1146, 1190, 1194, 1209, 1213, 1219, 1241, 1248, 1264, 1277, 1284, 1287, 1294, 1297, 1304, 1307, 1314, 1317, 1324,
    1327, 1334, 1337, 1344, 1347, 1354, 1357, 1364, 1367, 1382, 1382, 1414, 1419, 1451, 1455, 1483, 1484, 1512, 1515,
    1543, 1561, 1589, 1596, 1625, 1639, 1669, 1681, 1710, 1713, 1742, 1746, 1753, 1758, 1771, 1771, 1794, 1847, 1857,
    1858, 1867, 1867, 1876, 1876, 1884, 1884, 1890, 1890, 1897, 1905, 1911, 1911, 1930, 1931, 1956, 1957, 1967, 1967,
    1982, 1982, 1997, 2001, 2016, 2026};

__device__ __forceinline__ bool qpack_is_static(uint32_t kind) { return kind == kQIndexedStatic || kind == kQNameRefStatic; }
// Lines that name a dynamic table entry (relative or post-base): refused in a section whose Required Insert Count is 0.
__device__ __forceinline__ bool qpack_is_dynamic(uint32_t kind) {
    return kind == kQIndexedDynamic || kind == kQIndexedPostBase || kind == kQNameRefDynamic || kind == kQNameRefPostBase;
}
// Prefix bits, first-octet flags and N bit of each field line.
__device__ __forceinline__ uint32_t qpack_prefix_bits(uint32_t kind) { return 0x3344466u >> (4 * kind) & 15; }  // 6 6 4 4 4 3 3
__device__ __forceinline__ uint8_t qpack_prefix_flags(uint32_t kind) {
    return (uint8_t)(0x200040501080C0ull >> (8 * kind));  // 0xC0 0x80 0x10 0x50 0x40 0x00 0x20
}
__device__ __forceinline__ uint8_t qpack_never_flag(uint32_t kind) {
    return (uint8_t)(0x10082020000000ull >> (8 * kind));  // - - - 0x20 0x20 0x08 0x10
}

// ---- decode: the structural walk -----------------------------------------------------------------------------
struct SectionField {
    uint8_t kind;
    bool never;                // the N bit (false for the indexed lines)
    bool complete;             // false: the field failed after its name literal; only that literal is reported
    bool name_lit, value_lit;  // which literals below were read in full
    bool name_huff, value_huff;
    uint64_t index;
    // literal payloads, relative to the section (separate fields, not an array: see BlockField)
    uint64_t name_pay, name_len, value_pay, value_len;
};

// One string literal whose length integer starts at p[pos] (prefix_bits wide, Huffman flag huff_mask in that octet):
// its payload, or the error a decoder meets inside it.
__device__ __forceinline__ int32_t qpack_skip_literal(const uint8_t *p, uint64_t end, uint64_t &pos, uint32_t prefix_bits,
                                                      uint8_t huff_mask, bool &huff, uint64_t &pay, uint64_t &len) {
    if (pos >= end) return kStatusShortBuffer;
    huff = (p[pos] & huff_mask) != 0;
    const int32_t st = hpack_read_int(p, end, pos, prefix_bits, len);
    if (st != kStatusOk) return st;
    if (len > end - pos) return kStatusShortBuffer;
    pay = pos;
    pos += len;
    return kStatusOk;
}

// The section prefix at p[0 ..): Encoded Required Insert Count, S bit, Delta Base; pos is where the lines start.
__device__ __forceinline__ int32_t qpack_read_prefix(const uint8_t *p, uint64_t size, uint64_t &pos, uint64_t &eic,
                                                     uint8_t &sign, uint64_t &delta) {
    pos = 0;
    if (size == 0) return kStatusShortBuffer;
    const int32_t st = hpack_read_int(p, size, pos, 8, eic);
    if (st != kStatusOk) return st;
    if (pos >= size) return kStatusShortBuffer;
    sign = p[pos] >> 7;
    return hpack_read_int(p, size, pos, 7, delta);
}

// Walks one section front to back (the visitor contract of hpack_walk_block): its prefix, then every field line read
// in full is visited. Returns the first structural error (the walk stops there) or kStatusOk. A static index >= 99
// is refused after its integer; a dynamic or post-base reference in a section whose Encoded Required Insert Count is
// 0 is refused at its first octet (every absolute index is below a Required Insert Count of 0).
template <typename Visit>
__device__ __forceinline__ int32_t qpack_walk_section(const uint8_t *p, uint64_t size, Visit &&visit) {
    uint64_t pos, eic, delta;
    uint8_t sign;
    int32_t st = qpack_read_prefix(p, size, pos, eic, sign, delta);
    if (st != kStatusOk) return st;
    while (pos < size) {
        const uint8_t b0 = p[pos];
        SectionField f;
        f.complete = true;
        f.name_lit = f.value_lit = f.name_huff = f.value_huff = false;
        f.index = 0;
        if (b0 & 0x80)
            f.kind = (b0 & 0x40) ? kQIndexedStatic : kQIndexedDynamic;
        else if (b0 & 0x40)
            f.kind = (b0 & 0x10) ? kQNameRefStatic : kQNameRefDynamic;
        else if (b0 & 0x20)
            f.kind = kQLiteralName;
        else
            f.kind = (b0 & 0x10) ? kQIndexedPostBase : kQNameRefPostBase;
        f.never = (b0 & qpack_never_flag(f.kind)) != 0;
        if (f.kind == kQLiteralName) {
            st = qpack_skip_literal(p, size, pos, 3, 0x08, f.name_huff, f.name_pay, f.name_len);
            f.name_lit = st == kStatusOk;
        } else if (eic == 0 && qpack_is_dynamic(f.kind)) {
            st = kStatusInvalidArgument;
        } else {
            st = hpack_read_int(p, size, pos, qpack_prefix_bits(f.kind), f.index);
            if (st == kStatusOk && qpack_is_static(f.kind) && f.index >= kQpackStaticEntries) st = kStatusInvalidArgument;
        }
        if (st == kStatusOk && f.kind >= kQNameRefStatic) {  // (the lines with a value literal)
            st = qpack_skip_literal(p, size, pos, 7, 0x80, f.value_huff, f.value_pay, f.value_len);
            f.value_lit = st == kStatusOk;
        }
        if (st != kStatusOk) {
            if (f.name_lit) {
                f.complete = false;
                visit(f);
            }
            return st;
        }
        visit(f);
    }
    return kStatusOk;
}

// A literal's size in the packed batch: re-framed as an RFC 7541 5.2 literal.
__device__ __forceinline__ uint64_t qpack_reframed_bytes(uint64_t len) { return hpack_int_bytes(len, 7) + len; }

// Pass 1, thread per section: fields and literals read before the first structural error (a failing field's name
// literal included), their re-framed octets, and that error.
__global__ void qpack_section_scan_kernel(uint64_t n, const uint8_t *in, const uint64_t *in_offsets, uint64_t *num_fields,
                                          uint64_t *num_lits, uint64_t *lit_bytes, int32_t *struct_status) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t a = in_offsets[b];
    uint64_t nf = 0, nl = 0, nbytes = 0;
    struct_status[b] = qpack_walk_section(in + a, in_offsets[b + 1] - a, [&](const SectionField &f) {
        nf += f.complete;
        nl += f.name_lit + f.value_lit;
        if (f.name_lit) nbytes += qpack_reframed_bytes(f.name_len);
        if (f.value_lit) nbytes += qpack_reframed_bytes(f.value_len);
    });
    num_fields[b] = nf;
    num_lits[b] = nl;
    lit_bytes[b] = nbytes;
}

// The literal spans of one walked line (or instruction) whose item starts at in[a]: literal l (payload offset into
// `in`, length << 1 | H, offset of the re-framed literal in the packed batch) for its name and then its value, those
// read in full; name and value receive their literal ids, or kNoLiteral.
__device__ __forceinline__ void qpack_split_literals(const SectionField &fd, uint64_t a, uint64_t &l, uint64_t &o,
                                                     uint64_t *lit_src, uint64_t *lit_len, uint64_t *lit_offsets,
                                                     uint64_t &name, uint64_t &value) {
    name = value = kNoLiteral;
    if (fd.name_lit) {
        name = l;
        lit_src[l] = a + fd.name_pay;
        lit_len[l] = fd.name_len << 1 | fd.name_huff;
        lit_offsets[l++] = o;
        o += qpack_reframed_bytes(fd.name_len);
    }
    if (fd.value_lit) {
        value = l;
        lit_src[l] = a + fd.value_pay;
        lit_len[l] = fd.value_len << 1 | fd.value_huff;
        lit_offsets[l++] = o;
        o += qpack_reframed_bytes(fd.value_len);
    }
}

// Pass 2, thread per section, the same walk: field records (kind with the N bit, index, section, the literal ids of
// name and value) in parsed order from field_base[b], and literals (payload offset into `in`, length << 1 | H, offset
// of the re-framed literal in the packed batch) from lit_base[b] / lit_byte_base[b].
__global__ void qpack_section_split_kernel(
    uint64_t n, const uint8_t *in, const uint64_t *in_offsets, const uint64_t *field_base, const uint64_t *lit_base,
    const uint64_t *lit_byte_base, uint8_t *f_kind, uint64_t *f_index, uint32_t *f_block, uint64_t *f_lits,
    uint64_t *lit_src, uint64_t *lit_len, uint64_t *lit_offsets) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t a = in_offsets[b];
    uint64_t f = field_base[b], l = lit_base[b], o = lit_byte_base[b];
    qpack_walk_section(in + a, in_offsets[b + 1] - a, [&](const SectionField &fd) {
        uint64_t name, value;
        qpack_split_literals(fd, a, l, o, lit_src, lit_len, lit_offsets, name, value);
        if (!fd.complete) return;
        f_kind[f] = fd.kind | (fd.never ? kQNeverBit : 0);
        f_index[f] = fd.index;
        f_block[f] = (uint32_t)b;
        f_lits[2 * f] = name;
        f_lits[2 * f + 1] = value;
        ++f;
    });
    if (b == n - 1) lit_offsets[l] = o;
}

// The literals, packed and re-framed for the literal decoder: every lane writes its literal's H bit and 7-bit-prefix
// length, then the warp copies the 32 payloads (warp_run_jobs).
__global__ void __launch_bounds__(256) qpack_lit_gather_kernel(
    uint64_t num_lits, const uint8_t *in, const uint64_t *lit_src, const uint64_t *lit_len, const uint64_t *lit_offsets,
    uint8_t *dst) {
    __shared__ MoveJob s_jobs[8][32];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint64_t l = ((uint64_t)blockIdx.x * 8 + warp) * 32 + lane;
    MoveJob job = {nullptr, nullptr, 0};
    if (l < num_lits) {
        const uint64_t len = lit_len[l] >> 1, o = lit_offsets[l];
        hpack_put_int(dst, o, kNoCap, len, 7, (lit_len[l] & 1) ? 0x80 : 0x00);
        job.src = in + lit_src[l];
        job.dst = dst + o + hpack_int_bytes(len, 7);
        job.len = len;
    }
    warp_run_jobs(s_jobs, job, warp, lane);
}

// Where one string of a parsed field comes from: its decoded literal, the static table, or nowhere (a dynamic or
// post-base reference: empty).
__device__ __forceinline__ void qpack_field_string(
    uint8_t kind, uint64_t index, uint64_t lit, uint32_t which, const uint8_t *dec, const uint64_t *dec_offsets,
    const uint8_t *&src, uint64_t &len) {
    src = nullptr;
    len = 0;
    kind &= 7;
    if (lit != kNoLiteral) {
        src = dec + dec_offsets[lit];
        len = dec_offsets[lit + 1] - dec_offsets[lit];
    } else if (index < kQpackStaticEntries && (kind == kQIndexedStatic || (kind == kQNameRefStatic && which == 0))) {
        const uint32_t e = 2 * (uint32_t)index + which;
        src = kQpackStaticBlob + kQpackStaticOff[e];
        len = kQpackStaticOff[e + 1] - kQpackStaticOff[e];
    }
}

// The string source of QPACK fields for hpack_compose_kernel.
struct QpackFieldStrings {
    __device__ static void get(uint8_t kind, uint64_t index, uint64_t lit, uint32_t which, const uint8_t *dec,
                               const uint64_t *dec_offsets, const uint8_t *&src, uint64_t &len) {
        qpack_field_string(kind, index, lit, which, dec, dec_offsets, src, len);
    }
};

// Thread per parsed field: the record (kind, index, N bit) and the lengths of its two strings.
__global__ void qpack_field_records_kernel(
    uint64_t num_parsed, const uint8_t *f_kind, const uint64_t *f_index, const uint32_t *f_block, const uint64_t *f_lits,
    const uint64_t *field_base, const int32_t *status, const uint64_t *field_offsets, uint64_t field_capacity,
    const uint8_t *dec, const uint64_t *dec_offsets, uint8_t *out_kind, uint64_t *out_index, uint8_t *out_never,
    uint64_t *str_lens) {
    const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= num_parsed) return;
    const uint64_t o = hpack_out_field(f, f_block, field_base, status, field_offsets, field_capacity);
    if (o == ~0ull) return;
    const uint8_t kind = f_kind[f];
    const uint64_t index = f_index[f];
    out_kind[o] = kind & 7;
    out_index[o] = index;
    out_never[o] = (kind & kQNeverBit) ? 1 : 0;
    for (uint32_t w = 0; w < 2; ++w) {
        const uint8_t *src;
        uint64_t len;
        qpack_field_string(kind, index, f_lits[2 * f + w], w, dec, dec_offsets, src, len);
        str_lens[2 * o + w] = len;
    }
}

// Thread per section: the prefix integers as on the wire, or 0 for a section with a non-zero status.
__global__ void qpack_section_prefix_kernel(uint64_t n, const uint8_t *in, const uint64_t *in_offsets, const int32_t *status,
                                            uint64_t *eic, uint8_t *sign, uint64_t *delta) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    uint64_t pos, e = 0, d = 0;
    uint8_t s = 0;
    if (status[b] == kStatusOk) qpack_read_prefix(in + in_offsets[b], in_offsets[b + 1] - in_offsets[b], pos, e, s, d);
    eic[b] = e;
    sign[b] = s;
    delta[b] = d;
}

// ---- encode ---------------------------------------------------------------------------------------------------
// Plan byte of a field: line kind in bits 0..2, the flags of hpack_blocks.cuh (kPlanNameLit, kPlanValueLit,
// kPlanSkip) and the N bit; plan_index holds the integer after the first-octet flags (for a literal name: the name
// payload's length).
constexpr uint8_t kQPlanNever = 64;

// Record f's name and value (strings[string_offsets[2f] .. string_offsets[2f + 2])) against Appendix A: name_match is
// the lowest entry with that name, exact the lowest with that name and value (kQpackStaticEntries: none).
__device__ __forceinline__ void qpack_static_match(const uint8_t *strings, const uint64_t *string_offsets, uint64_t f,
                                                   uint32_t &name_match, uint32_t &exact) {
    const uint64_t n0 = string_offsets[2 * f], v0 = string_offsets[2 * f + 1], v1 = string_offsets[2 * f + 2];
    const uint8_t *name = strings + n0, *value = strings + v0;
    const uint64_t name_len = v0 - n0, value_len = v1 - v0;
    name_match = exact = kQpackStaticEntries;
    for (uint32_t e = 0; e < kQpackStaticEntries && exact == kQpackStaticEntries; ++e) {
        const uint32_t s0 = kQpackStaticOff[2 * e], s1 = kQpackStaticOff[2 * e + 1], s2 = kQpackStaticOff[2 * e + 2];
        if (s1 - s0 != name_len || !hpack_bytes_equal(name, kQpackStaticBlob + s0, name_len)) continue;
        if (name_match == kQpackStaticEntries) name_match = e;
        if (s2 - s1 == value_len && hpack_bytes_equal(value, kQpackStaticBlob + s1, value_len)) exact = e;
    }
}

// Thread per field: the line and its size on the wire from the framed literals (framed_offsets: name of field f is
// framed item 2f, its value 2f + 1). field_kind == NULL: every field is kQAuto; else the caller's kind and
// field_index[f] as given (ignored for a literal name). Static indices >= 99, unknown kinds and integers that
// hpack_read_int refuses get kPlanSkip and length 0.
__global__ void qpack_field_plan_kernel(
    uint64_t num_fields, const uint8_t *strings, const uint64_t *string_offsets, const uint8_t *never_indexed,
    const uint8_t *field_kind, const uint64_t *field_index, const uint8_t *framed, const uint64_t *framed_offsets,
    uint8_t *plan, uint64_t *plan_index, uint64_t *field_lens) {
    const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= num_fields) return;
    const uint8_t kind = field_kind ? field_kind[f] : kQAuto;
    const bool never = never_indexed && never_indexed[f];
    uint8_t p;
    uint64_t index = 0;
    if (kind == kQAuto) {
        uint32_t name_match, exact;
        qpack_static_match(strings, string_offsets, f, name_match, exact);
        if (!never && exact < kQpackStaticEntries) {
            p = kQIndexedStatic;
            index = exact;
        } else if (name_match < kQpackStaticEntries) {
            p = kQNameRefStatic;
            index = name_match;
        } else {
            p = kQLiteralName;
        }
    } else if (kind < kQAuto) {
        p = kind;
        if (kind != kQLiteralName) index = field_index[f];
        if (qpack_is_static(kind) && index >= kQpackStaticEntries) p |= kPlanSkip;
    } else {
        p = kPlanSkip;
    }
    const uint32_t k = p & 7;
    if (k >= kQNameRefStatic) {
        p |= kPlanValueLit;
        if (never) p |= kQPlanNever;
    }
    uint64_t len = 0;
    if (!(p & kPlanSkip)) {
        if (k == kQLiteralName) {
            // the framed name's payload length becomes the 3-bit-prefix integer
            p |= kPlanNameLit;
            uint64_t pos = framed_offsets[2 * f];
            hpack_read_int(framed, framed_offsets[2 * f + 1], pos, 7, index);
            len = index;
        }
        const uint32_t int_len = hpack_int_bytes(index, qpack_prefix_bits(k));
        if (int_len > 10) p |= kPlanSkip;
        len += int_len;
        if (p & kPlanValueLit) len += framed_offsets[2 * f + 2] - framed_offsets[2 * f + 1];
    }
    plan[f] = p;
    plan_index[f] = index;
    field_lens[f] = p & kPlanSkip ? 0 : len;
}

// Thread per section, after the plan. eic == NULL (stateless): every section is valid and its prefix is 00 00
// (Required Insert Count 0, Base 0). Else (records) the prefix is the caller's, and a section is invalid when a field
// of it is marked kPlanSkip, a dynamic or post-base line comes with an Encoded Required Insert Count of 0, S is not 0
// or 1, or a prefix integer is one hpack_read_int refuses. An invalid section gets INVALID_ARGUMENT in status
// (optional), every field of it kPlanSkip and length 0, and sec_lens[b] = 0; a valid one its prefix plus its fields.
__global__ void qpack_section_size_kernel(uint64_t n, const uint64_t *field_offsets, const uint64_t *eic, const uint8_t *sign,
                                          const uint64_t *delta, uint8_t *plan, uint64_t *field_lens, int32_t *status,
                                          uint64_t *sec_lens) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t f0 = field_offsets[b], f1 = field_offsets[b + 1];
    bool ok = true;
    uint64_t size = 2;
    if (eic) {
        const uint64_t e = eic[b], d = delta[b];
        ok = sign[b] <= 1 && hpack_int_bytes(e, 8) <= 10 && hpack_int_bytes(d, 7) <= 10;
        for (uint64_t f = f0; f < f1 && ok; ++f) {
            const uint8_t p = plan[f];
            ok = !(p & kPlanSkip) && !(e == 0 && qpack_is_dynamic(p & 7));
        }
        size = hpack_int_bytes(e, 8) + hpack_int_bytes(d, 7);
    }
    if (status) status[b] = ok ? kStatusOk : kStatusInvalidArgument;
    if (!ok) {
        for (uint64_t f = f0; f < f1; ++f) {
            plan[f] |= kPlanSkip;
            field_lens[f] = 0;
        }
        sec_lens[b] = 0;
        return;
    }
    for (uint64_t f = f0; f < f1; ++f) size += field_lens[f];
    sec_lens[b] = size;
}

// Thread per section, after the scans of section sizes (out_offsets) and of field sizes (field_pos, over all
// fields): a valid section writes its prefix and moves its fields' positions from the field scan onto the wire,
// behind its prefix. Never writes at or after out + out_capacity.
__global__ void qpack_section_place_kernel(uint64_t n, const uint64_t *field_offsets, const uint64_t *eic, const uint8_t *sign,
                                           const uint64_t *delta, const uint64_t *out_offsets, uint64_t *field_pos,
                                           uint8_t *out, uint64_t out_capacity) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t o = out_offsets[b];
    if (out_offsets[b + 1] == o) return;  // (an invalid section: a valid one holds at least its prefix)
    uint64_t lines = o + 2;
    if (eic) {
        hpack_put_int(out, o, out_capacity, eic[b], 8, 0x00);
        lines = o + hpack_int_bytes(eic[b], 8);
        hpack_put_int(out, lines, out_capacity, delta[b], 7, (uint8_t)(sign[b] << 7));
        lines += hpack_int_bytes(delta[b], 7);
    } else {
        if (o < out_capacity) out[o] = 0x00;
        if (o + 1 < out_capacity) out[o + 1] = 0x00;
    }
    const uint64_t f0 = field_offsets[b], f1 = field_offsets[b + 1];
    if (f0 == f1) return;
    const uint64_t shift = lines - field_pos[f0];  // (unsigned: wraps when the wire position is the smaller one)
    for (uint64_t f = f0; f < f1; ++f) field_pos[f] += shift;
}

// The wire format of field lines for qpack_field_emit_kernel (qpack_instructions.cuh has the instructions'): prefix
// bits and first-octet flags per plan byte, and the H bit of a name literal, whose length takes the line's prefix.
struct QpackFieldLines {
    static constexpr uint8_t kNameHuff = 0x08;
    __device__ static uint32_t prefix_bits(uint32_t kind) { return qpack_prefix_bits(kind); }
    __device__ static uint8_t flags(uint8_t plan) {
        return qpack_prefix_flags(plan & 7) | ((plan & kQPlanNever) ? qpack_never_flag(plan & 7) : 0);
    }
};

// A warp takes 32 lines: every lane writes its line's first-octet flags and integer, then the warp copies the 32
// name payloads (re-framed: their H bit and prefix-integer length went into the first octet) and the 32 framed value
// literals. Lines marked kPlanSkip write nothing. Never writes at or after out + out_capacity. Lines says what the
// first octet holds (QpackFieldLines: field lines).
template <typename Lines>
__global__ void __launch_bounds__(256) qpack_field_emit_kernel(
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
        uint8_t flags = Lines::flags(p);
        if ((p & kPlanNameLit) && (framed[framed_offsets[2 * f]] & 0x80)) flags |= Lines::kNameHuff;
        const uint32_t prefix_bits = Lines::prefix_bits(kind);
        hpack_put_int(out, pos, out_capacity, index, prefix_bits, flags);
        pos += hpack_int_bytes(index, prefix_bits);
        if (p & kPlanNameLit) {
            name.src = framed + framed_offsets[2 * f + 1] - index;
            name.dst = out + pos;
            name.len = pos < out_capacity ? min(index, out_capacity - pos) : 0;
            pos += index;
        }
        if (p & kPlanValueLit) {
            const uint64_t a = framed_offsets[2 * f + 1], len = framed_offsets[2 * f + 2] - a;
            value.src = framed + a;
            value.dst = out + pos;
            value.len = pos < out_capacity ? min(len, out_capacity - pos) : 0;
        }
    }
    warp_run_jobs(s_jobs, name, warp, lane);
    __syncwarp();
    warp_run_jobs(s_jobs, value, warp, lane);
}

}  // namespace hb
