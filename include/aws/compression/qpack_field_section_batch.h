#ifndef AWS_COMPRESSION_QPACK_FIELD_SECTION_BATCH_H
#define AWS_COMPRESSION_QPACK_FIELD_SECTION_BATCH_H
/*
 * Batched QPACK field sections (RFC 9204 section 4.5 field lines, Appendix A static table) on the device: HTTP/3's
 * header compression beside the HPACK header blocks of hpack_header_block_batch.h. QPACK uses HPACK's Huffman code
 * and prefix integers (RFC 9204 4.1). Same context, same conventions: CSR batches with 64-bit offsets, packed output,
 * AWS_ERROR_SHORT_BUFFER meaning "offsets are complete: size and retry", host and _device entry points, no CPU
 * fallback (AWS_ERROR_COMPRESSION_DEVICE_FAILURE without a device). A host-pointer call first waits for the context's
 * device calls still in flight on other streams.
 *
 * The wire layer of a field section is stateless: its prefix, where each field line starts, its kind, its integers,
 * its literals and the static table (indices 0..98) are all read here. What a dynamic or post-base reference means,
 * and the Required Insert Count and Base behind the prefix, depend on the connection's dynamic table, which stays the
 * caller's: such references are reported, not resolved, and the records encoder writes the references the caller
 * chose.
 */
#include <aws/compression/hpack_string_batch.h>

AWS_PUSH_SANE_WARNING_LEVEL

/* The representation of one field line (RFC 9204 section 4.5). */
enum aws_qpack_field_kind {
    AWS_QPACK_FIELD_INDEXED_STATIC = 0,     /* 4.5.2  11xxxxxx  static index (6-bit prefix)                       */
    AWS_QPACK_FIELD_INDEXED_DYNAMIC = 1,    /* 4.5.2  10xxxxxx  relative index (6-bit prefix)                     */
    AWS_QPACK_FIELD_INDEXED_POST_BASE = 2,  /* 4.5.3  0001xxxx  post-base index (4-bit prefix)                    */
    AWS_QPACK_FIELD_NAME_REF_STATIC = 3,    /* 4.5.4  01N1xxxx  static name index (4-bit prefix), value literal   */
    AWS_QPACK_FIELD_NAME_REF_DYNAMIC = 4,   /* 4.5.4  01N0xxxx  relative name index (4-bit prefix), value literal */
    AWS_QPACK_FIELD_NAME_REF_POST_BASE = 5, /* 4.5.5  0000Nxxx  post-base name index (3-bit prefix), value        */
    AWS_QPACK_FIELD_LITERAL_NAME = 6,       /* 4.5.6  001NHxxx  name literal (3-bit length prefix), value literal */
    AWS_QPACK_FIELD_AUTO = 7,               /* encode records only: the stateless rules choose (no decode)        */
};

/*
 * n field sections, one header list each. Section i starts with the prefix (encoded_insert_count[i], base_sign[i],
 * delta_base[i]) and owns fields [field_offsets[i], field_offsets[i+1]); field f's name is strings[string_offsets[2f]
 * .. string_offsets[2f+1]) and its value strings[string_offsets[2f+1] .. string_offsets[2f+2]). Offsets do not
 * decrease; on the encode side field_offsets[0] and string_offsets[0] are 0 (AWS_ERROR_INVALID_ARGUMENT otherwise,
 * checked by the host entry point).
 */
struct aws_qpack_field_sections {
    size_t n;                       /* field sections */
    uint64_t *encoded_insert_count; /* n: the prefix's first integer exactly as on the wire (8-bit prefix); decode:
                                       written; encode records: read; encode: ignored */
    uint8_t *base_sign;             /* n: the S bit; as above */
    uint64_t *delta_base;           /* n: Delta Base (7-bit prefix); as above */
    uint64_t *field_offsets;        /* n + 1 */
    uint64_t field_capacity;        /* decode: entries available in field_kind, field_index, never_indexed (and
                                       2 * this + 1 in string_offsets) */
    uint8_t *field_kind;            /* decode: written (enum aws_qpack_field_kind); encode records: read; encode: ignored */
    uint64_t *field_index;          /* static index, relative index or post-base index; 0 for LITERAL_NAME. decode:
                                       written; encode records: read; encode: ignored */
    uint8_t *never_indexed;         /* the N bit per field. decode: written (0 for the INDEXED kinds); encode: optional
                                       (NULL = none) */
    uint8_t *strings;
    uint64_t strings_capacity;      /* decode: bytes available in strings; encode: ignored */
    uint64_t *string_offsets;       /* 2 * fields + 1 */
};

AWS_EXTERN_C_BEGIN

/*
 * n field sections in (section i is in[in_offsets[i] .. in_offsets[i+1])), n header lists out. The prefix arrays get
 * the wire values (the library cannot compute Required Insert Count or Base: they need MaxEntries and the insert count
 * of the caller's table; see RFC 9204 4.5.1); they are 0 for a section with a non-zero status. Every field line
 * becomes one field record: field_kind, field_index and never_indexed. Static references are resolved into bytes
 * (INDEXED_STATIC: name and value of Appendix A; NAME_REF_STATIC: the Appendix A name and the decoded value). Dynamic
 * and post-base references are not: the strings that would come from the dynamic table are empty and field_index
 * names the entry.
 *
 * status (optional, n) per section, the first error a front-to-back decoder meets:
 *     0                                      decoded (a section with a prefix and no field lines is valid and has no
 *                                            fields)
 *     AWS_ERROR_SHORT_BUFFER                 the section ends inside the prefix (an empty section included), inside
 *                                            an integer or inside a literal
 *     AWS_ERROR_INVALID_ARGUMENT             a static index >= 99 (read in full), a dynamic or post-base reference in
 *                                            a section whose encoded insert count is 0 (refused at the line's first
 *                                            octet), or an integer with more continuation octets than 62 bits need
 *     AWS_ERROR_COMPRESSION_UNKNOWN_SYMBOL   from a Huffman literal: the rules of aws_hpack_string_decode_batch
 *     AWS_ERROR_COMPRESSION_INVALID_PADDING
 * A section with a non-zero status has no fields. When a LITERAL_NAME line fails after its name literal was read in
 * full, that literal is still decoded, and its errors win: they come first in byte order.
 *
 * Capacities: field_offsets[0..n] and the prefix arrays are always written. If field_offsets[n] > field_capacity the
 * call fails with AWS_ERROR_SHORT_BUFFER and string_offsets is undefined; else, if string_offsets[2 * field_offsets[n]]
 * > strings_capacity, it fails with AWS_ERROR_SHORT_BUFFER and string_offsets is complete. Bounds that always hold (so
 * a device caller never needs to read sizes first), with in_size = in_offsets[n]:
 *     field_capacity   >= in_size        (every field line takes at least one octet)
 *     strings_capacity >= 69 * in_size   (the one-octet line 0xfa, static entry 58, is "strict-transport-security"
 *                                         "max-age=31536000; includesubdomains; preload", 69 octets; two-octet
 *                                         indices and a Huffman octet's 8/5 symbols stay below that)
 */
AWS_COMPRESSION_API
int aws_qpack_field_section_decode_batch(
    struct aws_huffman_batch_ctx *ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    struct aws_qpack_field_sections *out,
    int32_t *status);

/*
 * in->n header lists in, n field sections out (out[out_offsets[i] .. out_offsets[i+1]), out_offsets has n + 1
 * entries; AWS_ERROR_SHORT_BUFFER when out_offsets[n] > out_capacity). The encoder is stateless: every section starts
 * 00 00 (Required Insert Count 0, Base 0) and no line references the dynamic table. Per field:
 *     1. never_indexed[f]:                  NAME_REF_STATIC with N = 1 and the lowest static index whose name matches,
 *                                           else LITERAL_NAME with N = 1
 *     2. (name, value) is in Appendix A:    INDEXED_STATIC with the lowest such index
 *     3. the name is in Appendix A:         NAME_REF_STATIC with N = 0 and the lowest such index
 *     4. otherwise:                         LITERAL_NAME with N = 0
 * Name and value literals are framed by `mode`. Names are not validated.
 */
AWS_COMPRESSION_API
int aws_qpack_field_section_encode_batch(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_qpack_field_sections *in,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets);

/*
 * The encoder for a caller that keeps its own dynamic table: the prefix of section i is written from
 * encoded_insert_count[i], base_sign[i] and delta_base[i], and field f as (field_kind[f], field_index[f],
 * never_indexed[f]) says: the records aws_qpack_field_section_decode_batch writes (the three prefix arrays,
 * in->field_kind and in->field_index must not be NULL). The N bit is written for the kinds that carry one; the
 * field_index of LITERAL_NAME and the never_indexed of the INDEXED kinds are ignored. AUTO takes the rules of
 * aws_qpack_field_section_encode_batch. Indices are written as given, so encoding the records a decode returned gives
 * back the decoded section (with the same Huffman choices). Literals are framed by `mode`. The strings a line does
 * not send are ignored (empty strings, or Appendix A strings as a decode writes them, are both fine).
 *
 * status (optional, n) per section: 0, or AWS_ERROR_INVALID_ARGUMENT when the section holds a kind above AUTO, a
 * static index >= 99, a dynamic or post-base kind while its encoded_insert_count is 0, a base_sign other than 0 or 1,
 * or an integer a decoder refuses (over 9 continuation octets). An invalid section encodes to zero octets
 * (out_offsets[i + 1] == out_offsets[i]: it has no prefix either); the other sections are not affected. Offsets,
 * capacity and AWS_ERROR_SHORT_BUFFER are as in aws_qpack_field_section_encode_batch; status is complete in every
 * case the offsets are.
 */
AWS_COMPRESSION_API
int aws_qpack_field_section_encode_records_batch(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_qpack_field_sections *in,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    int32_t *status);

/*
 * The same with device pointers (every array of `out` / `in` and `in`, `in_offsets`, `status`, `out`, `out_offsets`
 * live on the device); work is enqueued on cuda_stream (NULL = the context's stream). The caller reads the offsets
 * to learn the sizes and checks them against its capacities; nothing is written past a capacity.
 *
 * decode: in_size == in_offsets[n]. The call waits once, after the structural pass, for three totals (fields,
 * literals, literal octets): the literal decoder's launch is sized from them.
 * encode, encode records: num_fields == in->field_offsets[in->n], strings_size == in->string_offsets[2 *
 * num_fields]; they do not wait and read nothing back.
 */
AWS_COMPRESSION_API
int aws_qpack_field_section_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    uint64_t in_size,
    struct aws_qpack_field_sections *out,
    int32_t *status,
    void *cuda_stream);

AWS_COMPRESSION_API
int aws_qpack_field_section_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_qpack_field_sections *in,
    uint64_t num_fields,
    uint64_t strings_size,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    void *cuda_stream);

AWS_COMPRESSION_API
int aws_qpack_field_section_encode_records_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_qpack_field_sections *in,
    uint64_t num_fields,
    uint64_t strings_size,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    int32_t *status,
    void *cuda_stream);

AWS_EXTERN_C_END
AWS_POP_SANE_WARNING_LEVEL

#endif /* AWS_COMPRESSION_QPACK_FIELD_SECTION_BATCH_H */
