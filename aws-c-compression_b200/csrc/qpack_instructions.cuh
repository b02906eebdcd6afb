// QPACK encoder- and decoder-stream instructions (RFC 9204 sections 4.3 and 4.4) around the field-section code of
// qpack_sections.cuh: the same integers, literals, static table and pipeline.
//
//     encoder stream   insert, static name     11xxxxxx   name index, 6-bit prefix, value literal
//                      insert, dynamic name    10xxxxxx   relative name index, 6-bit prefix, value literal
//                      insert, literal name    01Hxxxxx   name length, 5-bit prefix, name payload, value literal
//                      duplicate               000xxxxx   relative index, 5-bit prefix
//                      set capacity            001xxxxx   capacity, 5-bit prefix
//     decoder stream   section acknowledgment  1xxxxxxx   stream ID, 7-bit prefix
//                      stream cancellation     01xxxxxx   stream ID, 6-bit prefix
//                      insert count increment  00xxxxxx   increment, 6-bit prefix (0 is an error)
//
// A chunk is a piece of one stream and may end inside an instruction: the walk stops before it (a cut), and the chunk's
// consumed length ends at the last instruction read in full.
// Decode: the walk of qpack_sections.cuh (thread per chunk, twice), the literals gathered re-framed for the HPACK
// literal decoder, then the finish, records and compose kernels of hpack_blocks.cuh with this file's string source.
// Encode: names and values framed by the literal path; one thread per instruction plans it; one thread per chunk
// refuses a chunk with a refused instruction; qpack_field_emit_kernel writes the instructions (QpackInstructionLines).
#pragma once

#include "qpack_sections.cuh"

namespace hb {

enum : uint8_t {
    kIInsertStatic = 0,
    kIInsertDynamic = 1,
    kIInsertLiteral = 2,
    kIDuplicate = 3,
    kISetCapacity = 4,
    kISectionAck = 5,
    kIStreamCancel = 6,
    kICountIncrement = 7,
    kIInsertAuto = 8,  // encode only: a static name reference when the name is in Appendix A, else a literal name
};

// Prefix bits and first-octet flags of each instruction.
__device__ __forceinline__ uint32_t qpack_instruction_prefix_bits(uint32_t kind) {
    return 0x66755566u >> (4 * kind) & 15;  // 6 6 5 5 5 7 6 6
}
__device__ __forceinline__ uint8_t qpack_instruction_flags(uint32_t kind) {
    return (uint8_t)(0x00408020004080C0ull >> (8 * kind));  // 0xC0 0x80 0x40 0x00 0x20 0x80 0x40 0x00
}
// which: 0 the encoder stream, 1 the decoder stream.
__device__ __forceinline__ bool qpack_instruction_of(uint32_t kind, uint32_t which) {
    return kind < kIInsertAuto && (kind >= kISectionAck) == (which == 1);
}

// ---- decode: the structural walk -----------------------------------------------------------------------------
// Walks one chunk front to back (the visitor contract of qpack_walk_section; instructions are SectionField records
// with the N bit clear) and visits every instruction read in full. A cut (the chunk ends inside an instruction) is
// not an error: the walk stops before that instruction and reports nothing of it. consumed: the octets of the
// instructions read in full. Returns the first structural error (a static name index >= 99 read in full, an Insert
// Count Increment of 0, an integer hpack_read_int refuses) or kStatusOk.
template <typename Visit>
__device__ __forceinline__ int32_t qpack_walk_instructions(const uint8_t *p, uint64_t size, uint32_t which,
                                                           uint64_t &consumed, Visit &&visit) {
    uint64_t pos = 0;
    consumed = 0;
    while (pos < size) {
        const uint8_t b0 = p[pos];
        SectionField f;
        f.never = false;
        f.complete = true;
        f.name_lit = f.value_lit = f.name_huff = f.value_huff = false;
        f.index = 0;
        if (which == 0) {
            if (b0 & 0x80)
                f.kind = (b0 & 0x40) ? kIInsertStatic : kIInsertDynamic;
            else if (b0 & 0x40)
                f.kind = kIInsertLiteral;
            else
                f.kind = (b0 & 0x20) ? kISetCapacity : kIDuplicate;
        } else {
            f.kind = (b0 & 0x80) ? kISectionAck : ((b0 & 0x40) ? kIStreamCancel : kICountIncrement);
        }
        int32_t st;
        if (f.kind == kIInsertLiteral) {
            st = qpack_skip_literal(p, size, pos, 5, 0x20, f.name_huff, f.name_pay, f.name_len);
            f.name_lit = st == kStatusOk;
        } else {
            st = hpack_read_int(p, size, pos, qpack_instruction_prefix_bits(f.kind), f.index);
            if (st == kStatusOk && ((f.kind == kIInsertStatic && f.index >= kQpackStaticEntries) ||
                                    (f.kind == kICountIncrement && f.index == 0)))
                st = kStatusInvalidArgument;
        }
        if (st == kStatusOk && f.kind <= kIInsertLiteral) {  // (the inserts: a value literal)
            st = qpack_skip_literal(p, size, pos, 7, 0x80, f.value_huff, f.value_pay, f.value_len);
            f.value_lit = st == kStatusOk;
        }
        if (st == kStatusShortBuffer) return kStatusOk;  // a cut: the instruction comes again, whole, with the next chunk
        if (st != kStatusOk) {
            if (f.name_lit) {
                f.complete = false;
                visit(f);
            }
            return st;
        }
        visit(f);
        consumed = pos;
    }
    return kStatusOk;
}

// Pass 1, thread per chunk: instructions and literals read before the first structural error (a failing
// instruction's name literal included), their re-framed octets, the consumed length and that error.
__global__ void qpack_instruction_scan_kernel(uint64_t n, uint32_t which, const uint8_t *in, const uint64_t *in_offsets,
                                              uint64_t *num_instr, uint64_t *num_lits, uint64_t *lit_bytes,
                                              uint64_t *consumed, int32_t *struct_status) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t a = in_offsets[b];
    uint64_t ni = 0, nl = 0, nbytes = 0, used;
    struct_status[b] = qpack_walk_instructions(in + a, in_offsets[b + 1] - a, which, used, [&](const SectionField &f) {
        ni += f.complete;
        nl += f.name_lit + f.value_lit;
        if (f.name_lit) nbytes += qpack_reframed_bytes(f.name_len);
        if (f.value_lit) nbytes += qpack_reframed_bytes(f.value_len);
    });
    num_instr[b] = ni;
    num_lits[b] = nl;
    lit_bytes[b] = nbytes;
    consumed[b] = used;
}

// Pass 2, thread per chunk, the same walk: instruction records (kind, index, chunk, the literal ids of name and value)
// from instr_base[b], and literals in the layout of qpack_section_split_kernel from lit_base[b] / lit_byte_base[b].
__global__ void qpack_instruction_split_kernel(
    uint64_t n, uint32_t which, const uint8_t *in, const uint64_t *in_offsets, const uint64_t *instr_base,
    const uint64_t *lit_base, const uint64_t *lit_byte_base, uint8_t *f_kind, uint64_t *f_index, uint32_t *f_block,
    uint64_t *f_lits, uint64_t *lit_src, uint64_t *lit_len, uint64_t *lit_offsets) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t a = in_offsets[b];
    uint64_t f = instr_base[b], l = lit_base[b], o = lit_byte_base[b], used;
    qpack_walk_instructions(in + a, in_offsets[b + 1] - a, which, used, [&](const SectionField &fd) {
        uint64_t name, value;
        qpack_split_literals(fd, a, l, o, lit_src, lit_len, lit_offsets, name, value);
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

// The string source of instructions for hpack_field_records_kernel and hpack_compose_kernel: a decoded literal, the
// Appendix A name of a static name reference, or empty.
struct QpackInstructionStrings {
    __device__ static void get(uint8_t kind, uint64_t index, uint64_t lit, uint32_t which, const uint8_t *dec,
                               const uint64_t *dec_offsets, const uint8_t *&src, uint64_t &len) {
        src = nullptr;
        len = 0;
        if (lit != kNoLiteral) {
            src = dec + dec_offsets[lit];
            len = dec_offsets[lit + 1] - dec_offsets[lit];
        } else if (kind == kIInsertStatic && which == 0 && index < kQpackStaticEntries) {
            src = kQpackStaticBlob + kQpackStaticOff[2 * index];
            len = kQpackStaticOff[2 * index + 1] - kQpackStaticOff[2 * index];
        }
    }
};

// Thread per chunk, after hpack_block_finish_kernel: a failing chunk consumed nothing.
__global__ void qpack_instruction_consumed_kernel(uint64_t n, const int32_t *status, uint64_t *consumed) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b < n && status[b] != kStatusOk) consumed[b] = 0;
}

// ---- encode ---------------------------------------------------------------------------------------------------
// Thread per instruction: the instruction and its size on the wire from the framed literals (name of instruction f is
// framed item 2f, its value 2f + 1; which == 1 frames nothing and reads neither). Plan bytes as in
// qpack_field_plan_kernel, plan_index the integer after the first-octet flags (for a literal name: the name payload's
// length). A kind of the other stream, a kind above AUTO, a static index >= 99, an Insert Count Increment of 0 and
// an integer hpack_read_int refuses get kPlanSkip and length 0.
__global__ void qpack_instruction_plan_kernel(
    uint64_t num_instr, uint32_t which, const uint8_t *strings, const uint64_t *string_offsets, const uint8_t *kind_in,
    const uint64_t *index_in, const uint8_t *framed, const uint64_t *framed_offsets, uint8_t *plan, uint64_t *plan_index,
    uint64_t *lens) {
    const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= num_instr) return;
    const uint8_t kind = kind_in[f];
    uint8_t p;
    uint64_t index = 0;
    if (kind == kIInsertAuto && which == 0) {
        uint32_t name_match, exact;
        qpack_static_match(strings, string_offsets, f, name_match, exact);
        p = name_match < kQpackStaticEntries ? kIInsertStatic : kIInsertLiteral;
        index = name_match < kQpackStaticEntries ? name_match : 0;
    } else if (qpack_instruction_of(kind, which)) {
        p = kind;
        if (kind != kIInsertLiteral) index = index_in[f];
        if ((kind == kIInsertStatic && index >= kQpackStaticEntries) || (kind == kICountIncrement && index == 0))
            p |= kPlanSkip;
    } else {
        p = kPlanSkip;
    }
    const uint32_t k = p & 7;
    uint64_t len = 0;
    if (!(p & kPlanSkip)) {
        if (k <= kIInsertLiteral) p |= kPlanValueLit;
        if (k == kIInsertLiteral) {
            // the framed name's payload length becomes the 5-bit-prefix integer
            p |= kPlanNameLit;
            uint64_t pos = framed_offsets[2 * f];
            hpack_read_int(framed, framed_offsets[2 * f + 1], pos, 7, index);
            len = index;
        }
        const uint32_t int_len = hpack_int_bytes(index, qpack_instruction_prefix_bits(k));
        if (int_len > 10) p |= kPlanSkip;
        len += int_len;
        if (p & kPlanValueLit) len += framed_offsets[2 * f + 2] - framed_offsets[2 * f + 1];
    }
    plan[f] = p;
    plan_index[f] = index;
    lens[f] = p & kPlanSkip ? 0 : len;
}

// Thread per chunk, after the plan and before the scan of instruction sizes: a chunk with an instruction marked
// kPlanSkip is invalid; it gets INVALID_ARGUMENT in status (optional) and every instruction of it kPlanSkip and
// length 0, so it encodes to zero octets.
__global__ void qpack_instruction_check_kernel(uint64_t n, const uint64_t *instruction_offsets, uint8_t *plan,
                                               uint64_t *lens, int32_t *status) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint64_t f0 = instruction_offsets[b], f1 = instruction_offsets[b + 1];
    bool ok = true;
    for (uint64_t f = f0; f < f1 && ok; ++f) ok = !(plan[f] & kPlanSkip);
    if (status) status[b] = ok ? kStatusOk : kStatusInvalidArgument;
    if (ok) return;
    for (uint64_t f = f0; f < f1; ++f) {
        plan[f] |= kPlanSkip;
        lens[f] = 0;
    }
}

// The wire format of instructions for qpack_field_emit_kernel: a literal name's H bit is 0x20 and its length takes the
// 5-bit prefix of INSERT_LITERAL_NAME.
struct QpackInstructionLines {
    static constexpr uint8_t kNameHuff = 0x20;
    __device__ static uint32_t prefix_bits(uint32_t kind) { return qpack_instruction_prefix_bits(kind); }
    __device__ static uint8_t flags(uint8_t plan) { return qpack_instruction_flags(plan & 7); }
};

}  // namespace hb
