#ifndef AWS_COMPRESSION_HPACK_HEADER_BLOCK_BATCH_H
#define AWS_COMPRESSION_HPACK_HEADER_BLOCK_BATCH_H
/*
 * Batched HPACK header blocks (RFC 7541 section 6 representations, Appendix A static table) on the device: the
 * layer above the string literals of hpack_string_batch.h. Same context, same conventions: CSR batches with 64-bit
 * offsets, packed output, AWS_ERROR_SHORT_BUFFER meaning "offsets are complete: size and retry", host and _device
 * entry points, no CPU fallback (AWS_ERROR_COMPRESSION_DEVICE_FAILURE without a device). A host-pointer call first
 * waits for the context's device calls still in flight on other streams.
 *
 * The wire layer of a header block is stateless: where each representation starts, its kind, its integers, its
 * literals and the static table (indices 1..61) are all read here. Only the meaning of an index >= 62 depends on
 * the connection's dynamic table, which stays the caller's: such references are reported, not resolved, and the
 * records encoder writes the references and insertions the caller chose.
 */
#include <aws/compression/hpack_string_batch.h>

AWS_PUSH_SANE_WARNING_LEVEL

/* The representation of one field (RFC 7541 section 6). */
enum aws_hpack_field_kind {
    AWS_HPACK_FIELD_INDEXED = 0,                  /* 6.1   1xxxxxxx: index (7-bit prefix)                       */
    AWS_HPACK_FIELD_LITERAL_INCREMENTAL = 1,      /* 6.2.1 01xxxxxx: name index (6-bit prefix, 0 = literal name) */
    AWS_HPACK_FIELD_LITERAL_WITHOUT_INDEXING = 2, /* 6.2.2 0000xxxx: name index (4-bit prefix)                  */
    AWS_HPACK_FIELD_LITERAL_NEVER_INDEXED = 3,    /* 6.2.3 0001xxxx: name index (4-bit prefix)                  */
    AWS_HPACK_FIELD_TABLE_SIZE_UPDATE = 4,        /* 6.3   001xxxxx: new maximum size (5-bit prefix)            */
    AWS_HPACK_FIELD_AUTO = 5,                     /* encode records only: the stateless rules choose (no decode) */
};

/*
 * n header lists, one per header block. List i owns fields [field_offsets[i], field_offsets[i+1]); field f's name
 * is strings[string_offsets[2f] .. string_offsets[2f+1]) and its value strings[string_offsets[2f+1] ..
 * string_offsets[2f+2]). Offsets do not decrease; on the encode side field_offsets[0] and string_offsets[0] are 0
 * (AWS_ERROR_INVALID_ARGUMENT otherwise, checked by the host entry point).
 */
struct aws_hpack_header_lists {
    size_t n;                  /* header blocks / lists */
    uint64_t *field_offsets;   /* n + 1 */
    uint64_t field_capacity;   /* decode: entries available in field_kind, field_index (and 2 * this + 1 in
                                  string_offsets) */
    uint8_t *field_kind;       /* decode: written (enum aws_hpack_field_kind); encode records: read; encode: ignored */
    uint64_t *field_index;     /* decode: written; encode records: read; encode: ignored */
    uint8_t *never_indexed;    /* encode: optional (NULL = none), one flag per field: sensitive fields (7.1.3) */
    uint8_t *strings;
    uint64_t strings_capacity; /* decode: bytes available in strings; encode: ignored */
    uint64_t *string_offsets;  /* 2 * fields + 1 */
};

AWS_EXTERN_C_BEGIN

/*
 * n header blocks in (block i is in[in_offsets[i] .. in_offsets[i+1])), n header lists out. Every representation
 * becomes one field record: field_kind and field_index, where field_index is
 *     INDEXED             the table index
 *     LITERAL_*           the name index (0: the name was a literal)
 *     TABLE_SIZE_UPDATE   the new maximum size
 * Static references (1..61) are resolved into bytes (INDEXED: name and value of Appendix A; a literal with an
 * indexed name: the Appendix A name and the decoded value). Dynamic references (>= 62) are not: the strings that
 * would come from the dynamic table are empty and field_index names the entry. LITERAL_INCREMENTAL fields are what
 * the caller inserts into its dynamic table; a TABLE_SIZE_UPDATE record has empty strings.
 *
 * status (optional, n) per block, the first error a front-to-back decoder meets:
 *     0                                      decoded (an empty block is valid and has no fields)
 *     AWS_ERROR_SHORT_BUFFER                 the block ends inside an integer or inside a literal
 *     AWS_ERROR_INVALID_ARGUMENT             index 0 in an indexed field, an integer with more continuation octets
 *                                            than 62 bits need, or a size update after the first field
 *     AWS_ERROR_COMPRESSION_UNKNOWN_SYMBOL   from a Huffman literal: the rules of aws_hpack_string_decode_batch
 *     AWS_ERROR_COMPRESSION_INVALID_PADDING
 * A block with a non-zero status has no fields.
 *
 * Capacities: field_offsets[0..n] is always written. If field_offsets[n] > field_capacity the call fails with
 * AWS_ERROR_SHORT_BUFFER and string_offsets is undefined; else, if string_offsets[2 * field_offsets[n]] >
 * strings_capacity, it fails with AWS_ERROR_SHORT_BUFFER and string_offsets is complete. Bounds that always hold
 * (so a device caller never needs to read sizes first), with in_size = in_offsets[n]:
 *     field_capacity   >= in_size        (every representation takes at least one octet)
 *     strings_capacity >= 28 * in_size   (the one-octet field 0x90 is "accept-encoding" "gzip, deflate", 28
 *                                         octets; a Huffman octet yields at most 8/5 symbols)
 */
AWS_COMPRESSION_API
int aws_hpack_header_block_decode_batch(
    struct aws_huffman_batch_ctx *ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    struct aws_hpack_header_lists *out,
    int32_t *status);

/*
 * in->n header lists in, n header blocks out (out[out_offsets[i] .. out_offsets[i+1]), out_offsets has n + 1
 * entries; AWS_ERROR_SHORT_BUFFER when out_offsets[n] > out_capacity). The encoder is stateless (it never inserts
 * into the dynamic table and never emits INCREMENTAL or a size update), and per field:
 *     1. never_indexed[f]:                  6.2.3, with the lowest static index whose name matches, else 0 and a
 *                                           name literal
 *     2. (name, value) is in Appendix A:    6.1 with that index
 *     3. the name is in Appendix A:         6.2.2 with the lowest such index
 *     4. otherwise:                         6.2.2 with index 0, a name literal and a value literal
 * Literals are framed by `mode` (names and values alike). Names are not validated.
 */
AWS_COMPRESSION_API
int aws_hpack_header_block_encode_batch(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_hpack_header_lists *in,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets);

/*
 * The encoder for a caller that keeps its own dynamic table: field f is written as the record (field_kind[f],
 * field_index[f]) says, the records aws_hpack_header_block_decode_batch writes (in->field_kind and in->field_index
 * must not be NULL). Per field_kind[f]:
 *     INDEXED                    6.1   1xxxxxxx  field_index (static or dynamic; 0 is invalid)
 *     LITERAL_INCREMENTAL        6.2.1 01xxxxxx  name index field_index (0: the name follows as a literal), value
 *     LITERAL_WITHOUT_INDEXING   6.2.2 0000xxxx  as above
 *     LITERAL_NEVER_INDEXED      6.2.3 0001xxxx  as above
 *     TABLE_SIZE_UPDATE          6.3   001xxxxx  field_index is the new maximum size
 *     AUTO                       the rules of aws_hpack_header_block_encode_batch, never_indexed[f] included;
 *                                field_index is ignored
 * Indices are written as given: there is no static lookup for an explicit kind, so encoding the records a decode
 * returned gives back the decoded block (with the same Huffman choices). The caller decides which fields enter its
 * table (INCREMENTAL) and when its size changes; the device does the octets. Literals are framed by `mode`. The
 * strings a representation does not send are ignored (the name and value of INDEXED and TABLE_SIZE_UPDATE, the name
 * behind a non-zero name index): empty strings, or Appendix A strings as a decode writes them, are both fine.
 *
 * status (optional, n) per block: 0, or AWS_ERROR_INVALID_ARGUMENT when the block holds a kind above AUTO, INDEXED
 * with index 0, a TABLE_SIZE_UPDATE after a field that is not one, or an integer a decoder refuses (over 9
 * continuation octets, i.e. at or above 2^63 plus the prefix's maximum). An invalid block encodes to zero octets
 * (out_offsets[i + 1] == out_offsets[i]); the other blocks are not affected. Offsets, capacity and
 * AWS_ERROR_SHORT_BUFFER are as in aws_hpack_header_block_encode_batch; status is complete in every case the
 * offsets are.
 */
AWS_COMPRESSION_API
int aws_hpack_header_block_encode_records_batch(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_hpack_header_lists *in,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    int32_t *status);

/*
 * The three calls above over several contexts, normally one per GPU of the box (contexts on the same device are
 * allowed; all of them made from the same code table, none used elsewhere during the call). The blocks or lists are
 * cut into n_ctx contiguous ranges balanced by octets (aws_huffman_batch_plan_shards): decode by block octets, encode
 * by the lists' string octets. Each range is staged from the caller's arrays, runs on its context on a host thread of
 * its own, and its records, offsets, status and octets are copied into place in the caller's arrays once every range
 * knows its bases. The return value, the error and every array written are those of the single-context call on
 * ctxs[0]: on AWS_ERROR_SHORT_BUFFER the offsets and status the rules above call complete are equal, and nothing is
 * written past a capacity. A failure in several ranges reports the first range's error. n_ctx == 1 is that call.
 * Errors of their own: AWS_ERROR_INVALID_ARGUMENT for ctxs == NULL, n_ctx == 0 or a NULL context.
 */
AWS_COMPRESSION_API
int aws_hpack_header_block_decode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs,
    size_t n_ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    struct aws_hpack_header_lists *out,
    int32_t *status);

AWS_COMPRESSION_API
int aws_hpack_header_block_encode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs,
    size_t n_ctx,
    const struct aws_hpack_header_lists *in,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets);

AWS_COMPRESSION_API
int aws_hpack_header_block_encode_records_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs,
    size_t n_ctx,
    const struct aws_hpack_header_lists *in,
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
int aws_hpack_header_block_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    uint64_t in_size,
    struct aws_hpack_header_lists *out,
    int32_t *status,
    void *cuda_stream);

AWS_COMPRESSION_API
int aws_hpack_header_block_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_hpack_header_lists *in,
    uint64_t num_fields,
    uint64_t strings_size,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    void *cuda_stream);

AWS_COMPRESSION_API
int aws_hpack_header_block_encode_records_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_hpack_header_lists *in,
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

#endif /* AWS_COMPRESSION_HPACK_HEADER_BLOCK_BATCH_H */
