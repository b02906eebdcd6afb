#ifndef AWS_COMPRESSION_QPACK_INSTRUCTION_BATCH_H
#define AWS_COMPRESSION_QPACK_INSTRUCTION_BATCH_H
/*
 * Batched QPACK encoder- and decoder-stream instructions (RFC 9204 sections 4.3 and 4.4) on the device: the two
 * unidirectional streams beside the field sections of qpack_field_section_batch.h. Same context, same conventions:
 * CSR batches with 64-bit offsets, packed output, AWS_ERROR_SHORT_BUFFER meaning "offsets are complete: size and
 * retry", host and _device entry points, no CPU fallback (AWS_ERROR_COMPRESSION_DEVICE_FAILURE without a device). A
 * host-pointer call first waits for the context's device calls still in flight on other streams.
 *
 * The wire layer of the instructions is stateless: where each instruction starts, its kind, its integers, its
 * literals and the static table (indices 0..98) are all read here. The dynamic table, its eviction, the check of a
 * capacity against SETTINGS_QPACK_MAX_TABLE_CAPACITY and the Required Insert Count / Base arithmetic stay the
 * caller's: instructions are reported, not applied.
 */
#include <aws/compression/qpack_field_section_batch.h>

AWS_PUSH_SANE_WARNING_LEVEL

/* Which stream a batch belongs to: the first-octet patterns of the two overlap. */
enum aws_qpack_instruction_stream {
    AWS_QPACK_ENCODER_STREAM = 0,
    AWS_QPACK_DECODER_STREAM = 1,
};

/* One instruction (RFC 9204 sections 4.3, 4.4). */
enum aws_qpack_instruction_kind {
    AWS_QPACK_INSERT_NAME_REF_STATIC = 0,  /* 4.3.2 11xxxxxx static name index (6-bit prefix), value literal     */
    AWS_QPACK_INSERT_NAME_REF_DYNAMIC = 1, /* 4.3.2 10xxxxxx relative name index (6-bit prefix), value literal   */
    AWS_QPACK_INSERT_LITERAL_NAME = 2,     /* 4.3.3 01Hxxxxx name literal (5-bit length prefix), value literal   */
    AWS_QPACK_DUPLICATE = 3,               /* 4.3.4 000xxxxx relative index (5-bit prefix)                       */
    AWS_QPACK_SET_CAPACITY = 4,            /* 4.3.1 001xxxxx capacity (5-bit prefix)                             */
    AWS_QPACK_SECTION_ACKNOWLEDGMENT = 5,  /* 4.4.1 1xxxxxxx stream ID (7-bit prefix)                            */
    AWS_QPACK_STREAM_CANCELLATION = 6,     /* 4.4.2 01xxxxxx stream ID (6-bit prefix)                            */
    AWS_QPACK_INSERT_COUNT_INCREMENT = 7,  /* 4.4.3 00xxxxxx increment (6-bit prefix); 0 is an error             */
    AWS_QPACK_INSERT_AUTO = 8,             /* encode only: static name ref if the name is in Appendix A, else
                                              literal name                                                       */
};

/*
 * n chunks of one stream's instructions. Chunk i owns instructions [instruction_offsets[i], instruction_offsets[i+1]);
 * instruction f's name is strings[string_offsets[2f] .. string_offsets[2f+1]) and its value strings[string_offsets[2f+1]
 * .. string_offsets[2f+2]). Offsets do not decrease; on the encode side instruction_offsets[0] and string_offsets[0]
 * are 0 (AWS_ERROR_INVALID_ARGUMENT otherwise, checked by the host entry point).
 */
struct aws_qpack_instructions {
    size_t n;                      /* chunks: one stream's octets each */
    uint64_t *instruction_offsets; /* n + 1 */
    uint64_t instruction_capacity; /* decode: entries available in kind, index (and 2 * this + 1 in string_offsets) */
    uint8_t *kind;                 /* enum aws_qpack_instruction_kind; decode: written, encode: read */
    uint64_t *index;               /* name index, relative index, capacity, stream ID or increment; 0 for a literal
                                      name. decode: written; encode: read (ignored for LITERAL_NAME and AUTO) */
    uint8_t *strings;
    uint64_t strings_capacity;     /* decode: bytes available in strings; encode: ignored */
    uint64_t *string_offsets;      /* 2 * instructions + 1: name, value per instruction (encode, decoder stream:
                                      ignored, may be NULL) */
};

AWS_EXTERN_C_BEGIN

/*
 * n chunks in (chunk i is in[in_offsets[i] .. in_offsets[i+1])), all from the stream `which`. Stream data arrives in
 * arbitrary pieces, so a chunk may end inside an instruction; that is not an error. Every instruction read in full
 * becomes one record (kind, index), and consumed[i] (n, required) is the octet count of chunk i's complete
 * instructions: the caller keeps the rest of the chunk and puts it in front of the next chunk of that stream. The cut
 * instruction yields nothing, and its name literal is not decoded even when that literal is complete: it is read
 * again in full. Strings per record:
 *     INSERT_NAME_REF_STATIC    the Appendix A name and the decoded value
 *     INSERT_NAME_REF_DYNAMIC   an empty name and the decoded value (index names the entry)
 *     INSERT_LITERAL_NAME       both decoded
 *     every other kind          both empty
 *
 * status (optional, n) per chunk, the first error a front-to-back decoder meets:
 *     0                                      decoded (the chunk may have ended inside an instruction)
 *     AWS_ERROR_INVALID_ARGUMENT             a static name index >= 99 (read in full), an integer with more
 *                                            continuation octets than 62 bits need, or an Insert Count Increment of 0
 *     AWS_ERROR_COMPRESSION_UNKNOWN_SYMBOL   from a Huffman literal: the rules of aws_hpack_string_decode_batch
 *     AWS_ERROR_COMPRESSION_INVALID_PADDING
 * When an INSERT_LITERAL_NAME fails structurally after its name literal was read in full, that literal is still
 * decoded, and its errors win: they come first in byte order (a cut is not a failure). A chunk with a non-zero status
 * has no instructions and consumed = 0: these are connection errors (QPACK_ENCODER_STREAM_ERROR or
 * QPACK_DECODER_STREAM_ERROR), after which nothing of the stream needs to survive.
 *
 * Capacities: instruction_offsets[0..n], consumed and status are always written. If instruction_offsets[n] >
 * instruction_capacity the call fails with AWS_ERROR_SHORT_BUFFER and string_offsets is undefined; else, if
 * string_offsets[2 * instruction_offsets[n]] > strings_capacity, it fails with AWS_ERROR_SHORT_BUFFER and
 * string_offsets is complete. Bounds that always hold, with in_size = in_offsets[n]:
 *     instruction_capacity >= in_size        (every instruction takes at least one octet)
 *     strings_capacity     >= 14 * in_size   (the two-octet insert e1 00, static name 33 "access-control-allow-headers"
 *                                             with an empty value, yields 28 octets; two-octet static indices and a
 *                                             Huffman octet's 8/5 symbols stay below that)
 * On the decoder stream every string is empty: strings may be NULL and strings_capacity 0.
 */
AWS_COMPRESSION_API
int aws_qpack_instruction_decode_batch(
    struct aws_huffman_batch_ctx *ctx,
    enum aws_qpack_instruction_stream which,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    struct aws_qpack_instructions *out,
    uint64_t *consumed,
    int32_t *status);

/*
 * in->n chunks of instructions in, n chunks of the stream `which` out (out[out_offsets[i] .. out_offsets[i+1]),
 * out_offsets has n + 1 entries; AWS_ERROR_SHORT_BUFFER when out_offsets[n] > out_capacity). The instructions are
 * written as kind and index say, so encoding the records a decode returned gives back the consumed octets (with the
 * same Huffman choices). INSERT_AUTO (encoder stream only) takes the lowest static index whose name matches, else a
 * literal name; its index is ignored. Literals are framed by `mode`; a literal name is re-framed into the 5-bit prefix
 * with H at 0x20. The strings a kind does not send are ignored.
 *
 * status (optional, n) per chunk: 0, or AWS_ERROR_INVALID_ARGUMENT when the chunk holds a kind of the other stream, a
 * kind above AUTO, a static index >= 99, an Insert Count Increment of 0, or an integer a decoder refuses (over 9
 * continuation octets). An invalid chunk encodes to zero octets; the other chunks are not affected. Offsets, capacity
 * and AWS_ERROR_SHORT_BUFFER are as in aws_qpack_field_section_encode_records_batch; status is complete in every case
 * the offsets are.
 */
AWS_COMPRESSION_API
int aws_qpack_instruction_encode_batch(
    struct aws_huffman_batch_ctx *ctx,
    enum aws_qpack_instruction_stream which,
    const struct aws_qpack_instructions *in,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    int32_t *status);

/*
 * The same with device pointers (every array of `out` / `in` and `in`, `in_offsets`, `consumed`, `status`, `out`,
 * `out_offsets` live on the device); work is enqueued on cuda_stream (NULL = the context's stream). The caller reads
 * the offsets to learn the sizes and checks them against its capacities; nothing is written past a capacity.
 *
 * decode: in_size == in_offsets[n]. The call waits once, after the structural pass, for three totals (instructions,
 * literals, literal octets): the literal decoder's launch is sized from them.
 * encode: num_instructions == in->instruction_offsets[in->n], strings_size == in->string_offsets[2 *
 * num_instructions] (0 on the decoder stream); it does not wait and reads nothing back.
 */
AWS_COMPRESSION_API
int aws_qpack_instruction_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    enum aws_qpack_instruction_stream which,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    uint64_t in_size,
    struct aws_qpack_instructions *out,
    uint64_t *consumed,
    int32_t *status,
    void *cuda_stream);

AWS_COMPRESSION_API
int aws_qpack_instruction_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    enum aws_qpack_instruction_stream which,
    const struct aws_qpack_instructions *in,
    uint64_t num_instructions,
    uint64_t strings_size,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    int32_t *status,
    void *cuda_stream);

AWS_EXTERN_C_END
AWS_POP_SANE_WARNING_LEVEL

#endif /* AWS_COMPRESSION_QPACK_INSTRUCTION_BATCH_H */
