#ifndef AWS_COMPRESSION_HPACK_STRING_BATCH_H
#define AWS_COMPRESSION_HPACK_STRING_BATCH_H
/*
 * Batched HPACK string literals (RFC 7541 section 5.2) on the device: the framing the immediate caller of
 * aws_huffman_encode / aws_huffman_decode puts around the codec (SURVEY.md 8f.1; in aws-c-http that caller is
 * the HPACK encoder / decoder, which picks the Huffman form by an aws_hpack_huffman_mode and validates the
 * padding with the decoder's leftover bits as the reference's README.md:176-183 describes). The reference
 * repository itself holds no framing code; behaviour is anchored on RFC 7541 sections 5.1 / 5.2 and its
 * Appendix C vectors (tests/test_hpack_literals.py).
 *
 *     | H | length (7-bit prefix integer, section 5.1) | length octets of string data |
 *
 * The context must have been created from the RFC 7541 Appendix B code (any prefix code works mechanically:
 * "EOS prefix" is taken to mean all ones, which is what HPACK's EOS is).
 * Strings and literals are CSR batches: item i is in[in_offsets[i] .. in_offsets[i+1]). Output is packed:
 * the calls write out_offsets[0..n]; if out_offsets[n] > out_capacity they fail with AWS_ERROR_SHORT_BUFFER
 * (offsets complete: size and retry). No CPU fallback: AWS_ERROR_COMPRESSION_DEVICE_FAILURE without a device.
 */
#include <aws/compression/huffman_batch.h>

AWS_PUSH_SANE_WARNING_LEVEL

/* How an encoder chooses between the raw and the Huffman form of a string (the choices of aws-c-http's
 * enum aws_hpack_huffman_mode). SMALLEST: Huffman only when strictly shorter. */
enum aws_hpack_huffman_mode {
    AWS_HPACK_HUFFMAN_SMALLEST = 0,
    AWS_HPACK_HUFFMAN_NEVER = 1,
    AWS_HPACK_HUFFMAN_ALWAYS = 2,
};

AWS_EXTERN_C_BEGIN

/* n strings in, n string literals out (H bit, length, payload). Host pointers. A host-pointer call first waits for
 * the context's device calls still in flight on other streams. */
AWS_COMPRESSION_API
int aws_hpack_string_encode_batch(
    struct aws_huffman_batch_ctx *ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets);

/*
 * n string literals in (item i is exactly one literal), n strings out. status (optional, n) per item:
 *     0                                      decoded
 *     AWS_ERROR_SHORT_BUFFER                 the literal is cut short: no length byte, an unfinished length, or
 *                                            fewer payload octets than the length announces
 *     AWS_ERROR_INVALID_ARGUMENT             octets left over after the payload, or a length beyond 2^62
 *     AWS_ERROR_COMPRESSION_UNKNOWN_SYMBOL   the Huffman payload holds a bit sequence that is no code (this is also how an
 *                                            EOS code with 32 bits or more of payload behind it reports: the decoder
 *                                            stops there, exactly like aws_huffman_decode)
 *     AWS_ERROR_COMPRESSION_INVALID_PADDING  padding of 8 bits or more, padding that is not all ones (an EOS code in the
 *                                            last 32 bits of the payload reports here: it is a run of ones too long)
 * Items with a non-zero status decode to nothing (their output range is empty).
 */
AWS_COMPRESSION_API
int aws_hpack_string_decode_batch(
    struct aws_huffman_batch_ctx *ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    int32_t *status);

/*
 * The same over several contexts, normally one per GPU of the box (contexts on the same device are allowed; all of
 * them made from the same code table, none used elsewhere during the call). The items are cut into n_ctx contiguous
 * ranges balanced by input octets (aws_huffman_batch_plan_shards); each range is staged from the caller's arrays, runs
 * on its context on a host thread of its own and is copied into place in the caller's arrays. The return value, the
 * error and every array written (out_offsets, out, status) are those of the single-context call on ctxs[0],
 * AWS_ERROR_SHORT_BUFFER included; a failure in several ranges reports the first range's error. n_ctx == 1 is that
 * call. Errors of their own: AWS_ERROR_INVALID_ARGUMENT for ctxs == NULL, n_ctx == 0 or a NULL context.
 */
AWS_COMPRESSION_API
int aws_hpack_string_encode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs,
    size_t n_ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets);

AWS_COMPRESSION_API
int aws_hpack_string_decode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs,
    size_t n_ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    int32_t *status);

/* The same with device pointers; work is enqueued on cuda_stream (NULL = the context's stream). in_size ==
 * in_offsets[n] (the offsets live on the device). The caller reads out_offsets[n] to learn the size. */
AWS_COMPRESSION_API
int aws_hpack_string_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    uint64_t in_size,
    enum aws_hpack_huffman_mode mode,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    void *cuda_stream);

AWS_COMPRESSION_API
int aws_hpack_string_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    size_t n,
    const uint8_t *in,
    const uint64_t *in_offsets,
    uint64_t in_size,
    uint8_t *out,
    uint64_t out_capacity,
    uint64_t *out_offsets,
    int32_t *status,
    void *cuda_stream);

AWS_EXTERN_C_END
AWS_POP_SANE_WARNING_LEVEL

#endif /* AWS_COMPRESSION_HPACK_STRING_BATCH_H */
