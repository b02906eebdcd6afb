#ifndef AWS_COMPRESSION_HUFFMAN_BATCH_H
#define AWS_COMPRESSION_HUFFMAN_BATCH_H
/*
 * Batched Huffman encode/decode on one NVIDIA B200 (sm_100a CUDA), behind a plain C ABI.
 *
 * These entry points do not exist in the reference; they are the GPU sibling of
 * aws_huffman_encode / aws_huffman_decode (reference include/aws/compression/huffman.h:133-152,
 * source/huffman.c:131-187,213-286). Contract per item i of a batch:
 *
 *     the bytes, lengths, status, consumed count and leftover state are exactly what ONE call of
 *     aws_huffman_encode (resp. aws_huffman_decode) returns on a freshly initialised
 *     aws_huffman_encoder (resp. aws_huffman_decoder) for the same coder, the same input and
 *     the item's output capacity.
 *
 * n == 1 with a large input is the "single long stream" case; the library picks chunked kernels
 * for long items by itself. There is no CPU fallback: without a usable device every call fails
 * with AWS_ERROR_COMPRESSION_DEVICE_FAILURE.
 *
 * Everything is plain pointers and sizes so that cgo / JNI / N-API / ctypes can bind it directly.
 */
#include <aws/compression/huffman.h>

AWS_PUSH_SANE_WARNING_LEVEL

/* Owns the device-side code table, decode lookup tables, a stream and scratch memory for one
 * (coder, eos_padding, device). Not re-entrant; use one context per calling thread. */
struct aws_huffman_batch_ctx;

/*
 * One batch. `in` / `in_offsets` describe n items back to back (CSR): item i is
 * in[in_offsets[i] .. in_offsets[i+1]). Two output layouts:
 *
 *   packed  (out_caps == NULL): results are written back to back; the call WRITES
 *           out_offsets[0..n] (exclusive prefix sum of out_lens; out_offsets[n] = bytes needed).
 *           Every item behaves as if it had all the room it needs, so per-item status is 0 or
 *           AWS_ERROR_COMPRESSION_UNKNOWN_SYMBOL. If out_offsets[n] > out_capacity the call
 *           fails with AWS_ERROR_SHORT_BUFFER (out_offsets is still complete: size and retry).
 *   slotted (out_caps != NULL): the call READS out_offsets[0..n-1]; item i is written at
 *           out + out_offsets[i] and may use out_caps[i] bytes; slots must not overlap. Per-item
 *           status may also be AWS_ERROR_SHORT_BUFFER, with `consumed`, `out_lens` and the
 *           leftover state telling where the reference would have stopped.
 *
 * Optional arrays may be NULL. For the *_device entry points every pointer is a device pointer.
 */
struct aws_huffman_batch {
    size_t n;
    const uint8_t *in;
    const uint64_t *in_offsets; /* n + 1 entries, non-decreasing, in_offsets[0] == 0 */
    uint64_t in_size;           /* == in_offsets[n]. The *_device entry points size their grids from it
                                 * (in_offsets lives on the device there); the host entry points ignore it. */

    uint8_t *out;
    uint64_t out_capacity;   /* bytes addressable at `out` */
    uint64_t *out_offsets;   /* n + 1 entries; written (packed) or read (slotted) */
    const uint64_t *out_caps; /* NULL = packed; else n per-item capacities */

    uint64_t *out_lens; /* optional, n: bytes written for item i (aws_byte_buf.len after the call) */
    int32_t *status;    /* optional, n: 0, AWS_ERROR_SHORT_BUFFER or AWS_ERROR_COMPRESSION_UNKNOWN_SYMBOL */
    uint64_t *consumed; /* optional, n: how far the input cursor advanced */

    /* encode only, optional, n each: encoder->overflow_bits after the call (pattern reported as 0
     * when num_bits is 0) */
    uint32_t *overflow_pattern;
    uint8_t *overflow_num_bits;

    /* decode only, optional, n each: decoder->working_bits / decoder->num_bits after the call
     * (what README.md:176-183 of the reference uses to validate HPACK padding) */
    uint64_t *leftover_working_bits;
    uint8_t *leftover_num_bits;
};

AWS_EXTERN_C_BEGIN

/*
 * Calls coder->encode once per symbol 0..255 on the host, checks the result is a prefix code,
 * and uploads the code table and the multi-level decode lookup tables to `device_id`.
 * Errors: AWS_ERROR_COMPRESSION_INVALID_CODE_TABLE, AWS_ERROR_COMPRESSION_DEVICE_FAILURE,
 * AWS_ERROR_OOM. The coder is not retained.
 */
AWS_COMPRESSION_API
int aws_huffman_batch_ctx_new(
    struct aws_huffman_batch_ctx **out_ctx,
    struct aws_huffman_symbol_coder *coder,
    uint8_t eos_padding,
    int device_id);

/*
 * The same from a raw 256-entry code table (num_bits == 0: the symbol has no code), e.g. the
 * <name>_get_code_table() that huffman_generator emits next to <name>_get_coder(): no callback is
 * ever called (SURVEY.md 8f.2: device-ready tables straight from the generator's output).
 */
AWS_COMPRESSION_API
int aws_huffman_batch_ctx_new_from_code_table(
    struct aws_huffman_batch_ctx **out_ctx,
    const struct aws_huffman_code *code_table,
    uint8_t eos_padding,
    int device_id);

AWS_COMPRESSION_API
void aws_huffman_batch_ctx_destroy(struct aws_huffman_batch_ctx *ctx);

/* Host buffers in, host buffers out (copies staged through the context's stream). A host-pointer call first waits
 * for the context's device calls still in flight on other streams. */
AWS_COMPRESSION_API
int aws_huffman_encode_batch(struct aws_huffman_batch_ctx *ctx, const struct aws_huffman_batch *batch);

AWS_COMPRESSION_API
int aws_huffman_decode_batch(struct aws_huffman_batch_ctx *ctx, const struct aws_huffman_batch *batch);

/*
 * Device buffers in, device buffers out. Work is enqueued on `cuda_stream` (a cudaStream_t; NULL
 * = the context's own stream) and the call returns without waiting unless scratch memory has to
 * grow. Writes never go past out + out_capacity. In packed layout the caller reads
 * out_offsets[n] itself to learn the size.
 */
AWS_COMPRESSION_API
int aws_huffman_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_huffman_batch *batch,
    void *cuda_stream);

AWS_COMPRESSION_API
int aws_huffman_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_huffman_batch *batch,
    void *cuda_stream);

/*
 * Streaming continuation (SURVEY.md 8f.3): the batched form of calling aws_huffman_encode /
 * aws_huffman_decode AGAIN on the same encoder / decoder, the way the reference is fed from network
 * buffers (tests/huffman_test.c:117-165 and :275-363, source/huffman_testing.c). Per item the state arrays
 * are read first and written afterwards, and they are required:
 *     encode: overflow_pattern[i] / overflow_num_bits[i]  = encoder->overflow_bits (source/huffman.c:150-160:
 *             written before the item's first symbol; left as they are when there is no room at all)
 *     decode: leftover_working_bits[i] / leftover_num_bits[i] = decoder->working_bits / num_bits
 *             (source/huffman.c:196-211,222)
 * Everything else is the contract above. Zeroed state arrays give exactly aws_huffman_encode_batch /
 * aws_huffman_decode_batch. A caller loops: items that returned AWS_ERROR_SHORT_BUFFER come back with
 * `in` advanced by consumed[i] and a fresh output slot; a decoder fed chunk by chunk comes back with the
 * next chunk. These calls run on the per-item kernels (every capacity rule in closed form), not on the
 * tiled throughput kernels.
 */
AWS_COMPRESSION_API
int aws_huffman_encode_batch_resume(struct aws_huffman_batch_ctx *ctx, const struct aws_huffman_batch *batch);

AWS_COMPRESSION_API
int aws_huffman_decode_batch_resume(struct aws_huffman_batch_ctx *ctx, const struct aws_huffman_batch *batch);

AWS_COMPRESSION_API
int aws_huffman_encode_batch_resume_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_huffman_batch *batch,
    void *cuda_stream);

AWS_COMPRESSION_API
int aws_huffman_decode_batch_resume_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_huffman_batch *batch,
    void *cuda_stream);

/* Batched aws_huffman_get_encoded_length (reference huffman.h:121, huffman.c:107-129):
 * lens[i] = ceil(sum of code lengths / 8), unknown symbols counting 0. Host pointers. */
AWS_COMPRESSION_API
int aws_huffman_get_encoded_length_batch(
    struct aws_huffman_batch_ctx *ctx,
    const uint8_t *in,
    const uint64_t *in_offsets,
    size_t n,
    uint64_t *lens);

/* The same with device pointers (reference huffman.c:107-129 per item); enqueued on `cuda_stream`
 * (NULL = the context's own stream), returns without waiting. */
AWS_COMPRESSION_API
int aws_huffman_get_encoded_length_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const uint8_t *in,
    const uint64_t *in_offsets,
    size_t n,
    uint64_t *lens,
    void *cuda_stream);

/* Blocks until everything enqueued on the context's own stream has finished. */
AWS_COMPRESSION_API
int aws_huffman_batch_ctx_synchronize(struct aws_huffman_batch_ctx *ctx);

/* The context's stream (cudaStream_t) and device ordinal, for callers that time or chain work. */
AWS_COMPRESSION_API
void *aws_huffman_batch_ctx_stream(struct aws_huffman_batch_ctx *ctx);
AWS_COMPRESSION_API
int aws_huffman_batch_ctx_device(struct aws_huffman_batch_ctx *ctx);

/* Kernels launched by this context since creation (bench.py's gpu_launches). */
AWS_COMPRESSION_API
uint64_t aws_huffman_batch_ctx_launch_count(struct aws_huffman_batch_ctx *ctx);

/*
 * Multi-GPU sharding helpers (host only, no device needed). Items are independent, so a batch is
 * split into contiguous index ranges balanced by input bytes, one range per GPU, with no
 * collective. shard_begin receives num_shards + 1 item indices.
 */
AWS_COMPRESSION_API
int aws_huffman_batch_plan_shards(const uint64_t *in_offsets, size_t n, size_t num_shards, size_t *shard_begin);

/* Rebases shard-local packed out_offsets (each starting at 0) into one global array of
 * total_items + 1 entries: the host-side concatenation step. shard_offsets[s] has
 * shard_items[s] + 1 entries. */
AWS_COMPRESSION_API
int aws_huffman_batch_concat_offsets(
    const uint64_t *const *shard_offsets,
    const size_t *shard_items,
    size_t num_shards,
    uint64_t *global_offsets);

/*
 * One packed batch over several contexts — normally one per GPU of the box (BASELINE configs[4]); contexts on
 * the same device are allowed. The batch is cut into n_ctx contiguous item ranges balanced by input bytes
 * (aws_huffman_batch_plan_shards), every range runs through its context's host path on a host thread of its own,
 * and payloads and offsets are concatenated on the host (aws_huffman_batch_concat_offsets). Per item the result is
 * exactly that of aws_huffman_encode_batch / aws_huffman_decode_batch on one context: the reference's
 * aws_huffman_encode / aws_huffman_decode (source/huffman.c:131-187, 213-286) per item. Host pointers, packed
 * layout only (out_caps must be NULL). All contexts must have been created from the same coder.
 */
AWS_COMPRESSION_API
int aws_huffman_encode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs,
    size_t n_ctx,
    const struct aws_huffman_batch *batch);

AWS_COMPRESSION_API
int aws_huffman_decode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs,
    size_t n_ctx,
    const struct aws_huffman_batch *batch);

AWS_EXTERN_C_END
AWS_POP_SANE_WARNING_LEVEL

#endif /* AWS_COMPRESSION_HUFFMAN_BATCH_H */
