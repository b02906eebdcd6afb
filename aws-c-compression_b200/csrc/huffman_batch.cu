// C-ABI of the batched Huffman codec (include/aws/compression/huffman_batch.h) and the host-side
// orchestration around the CUDA kernels: context (device tables, stream, scratch), host<->device
// staging for the host-pointer entry points, kernel selection and launch.
//
// No CPU fallback lives here: every failure to reach the device surfaces as
// AWS_ERROR_COMPRESSION_DEVICE_FAILURE.
#include <aws/compression/huffman_batch.h>
#include <aws/compression/hpack_string_batch.h>
#include <aws/compression/hpack_header_block_batch.h>
#include <aws/compression/qpack_field_section_batch.h>
#include <aws/compression/qpack_instruction_batch.h>
#include <aws/compression/huffman_table_builder.h>

#include "../host/huffman_lut.h"
#include "device_common.cuh"
#include "generic_kernels.cuh"
#include "encode_tiled.cuh"
#include "encode_slots.cuh"
#include "encode_strings.cuh"
#include "hpack_literals.cuh"
#include "hpack_blocks.cuh"
#include "qpack_sections.cuh"
#include "qpack_instructions.cuh"
#include "decode_fast.cuh"

#include <algorithm>
#include <array>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

namespace {

using namespace hb;

#define HB_CUDA_TRY(expr)                                                                                              \
    do {                                                                                                               \
        cudaError_t hb_err_ = (expr);                                                                                  \
        if (hb_err_ != cudaSuccess) {                                                                                  \
            hb_note_cuda_error(hb_err_, #expr, __LINE__);                                                              \
            return aws_raise_error(AWS_ERROR_COMPRESSION_DEVICE_FAILURE);                                              \
        }                                                                                                              \
    } while (0)

void hb_note_cuda_error(cudaError_t err, const char *what, int line) {
    if (getenv("AWS_HUFFMAN_BATCH_DEBUG")) {
        fprintf(stderr, "aws-c-compression(b200): %s failed at line %d: %s\n", what, line, cudaGetErrorString(err));
    }
    (void)cudaGetLastError(); /* clear the sticky-less error slot */
}

}  // namespace

namespace hb_host {
// Device buffer that only ever grows; freed with its owner.
struct GrowBuf {
    void *ptr = nullptr;
    size_t bytes = 0;

    GrowBuf() = default;
    GrowBuf(const GrowBuf &) = delete;
    GrowBuf &operator=(const GrowBuf &) = delete;
    ~GrowBuf() {
        if (ptr) cudaFree(ptr);
    }
    cudaError_t reserve(size_t want) {
        if (want <= bytes) return cudaSuccess;
        size_t grown = std::max(want, bytes + bytes / 2);
        grown = (grown + 255) & ~size_t(255);
        void *fresh = nullptr;
        cudaError_t err = cudaMalloc(&fresh, grown);
        if (err != cudaSuccess) return err;
        if (ptr) cudaFree(ptr);
        ptr = fresh;
        bytes = grown;
        return cudaSuccess;
    }
    template <typename T>
    T *as() const {
        return static_cast<T *>(ptr);
    }
};
// Per-launch kernel scratch (tile descriptors, chunk records, ...). One per concurrent stream.
struct Scratch {
    GrowBuf lens, tile_state, tile_first, chunks, chunk_lens, chunk_offsets, fused, slot_base, deferred, str_ctl, str_state,
        str_tiles, str_bits, str_bits_first;
};

// lanes of the pipelined host path (round 2, 12 MiB sub-batches: retired one issue later with 4 lanes 60.9,
// two issues later with 5 lanes 59.7, one issue later with 3 lanes 59.6 GB/s end to end)
constexpr size_t kLanes = 4;
struct Lane {
    cudaStream_t stream = nullptr;
    cudaEvent_t kernels_done = nullptr, retired = nullptr;
    bool in_flight = false;
    uint64_t *h_total = nullptr;  // pinned: the sub-batch's output size
    Scratch scratch;
    GrowBuf in, in_off, out, out_off, lens, status, consumed, aux32, aux8, aux64;
    ~Lane() {
        if (h_total) cudaFreeHost(h_total);
        if (kernels_done) cudaEventDestroy(kernels_done);
        if (retired) cudaEventDestroy(retired);
        if (stream) cudaStreamDestroy(stream);
    }
};
// HPACK header blocks (hpack_blocks.cuh) and QPACK field sections (qpack_sections.cuh): per-block counts and bases,
// parsed fields, literal spans and the decoded literals, encode plans, and the staging of the host entry points' extra
// arrays.
struct BlockBufs {
    GrowBuf num_fields, num_lits, lit_bytes, struct_status, out_fields, status, field_base, lit_base, lit_byte_base,
        f_kind, f_index, f_block, f_lits, lit_src, lit_offsets, lits, dec, dec_offsets, lit_status, str_lens, plan,
        plan_index, field_lens, field_pos, framed, framed_offsets, s_field_offsets, s_never, s_kind, s_index,
        s_string_offsets;
    GrowBuf lit_len, sec_lens, s_eic, s_sign, s_delta;  // QPACK only: literal lengths and H bits, section sizes, prefixes
    uint64_t *h_totals = nullptr;  // pinned: fields, literals, literal octets
    ~BlockBufs() {
        if (h_totals) cudaFreeHost(h_totals);
    }
};
// Shared-memory layout of decode_batch_kernel<framed> (decode_batch_fast): [LUT2][team 0: stage, rows][team 1: ...].
struct DecLayout {
    size_t stage_bytes = 0, rows_bytes = 0, smem = 0;
};
// Shared memory of the single-stream kernels (decode_stream_fast), and whether the fused kernel runs.
struct StreamLayout {
    uint32_t row_words = 0;
    size_t smem = 0, smem_staged = 0, fused_smem = 0;
    bool fused = false;
};
}  // namespace hb_host
using hb_host::GrowBuf;
using hb_host::Lane;
using hb_host::Scratch;

struct aws_huffman_batch_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    hb::DeviceTables tables{};
    uint2 *d_enc = nullptr;
    uint32_t *d_lut = nullptr;
    uint2 *d_lut2 = nullptr;  // 64-bit entries of the lean decode step (decode_fast.cuh)
    uint32_t lut2_count = 0, lut2_trap = 0;
    uint32_t lut_smem_entries = 0;
    uint64_t launches = 0;

    // kernel scratch for the device entry points (and the simple host path)
    hb_host::Scratch scratch;
    // pipelined host path: independent lanes (stream + scratch + staging) so that the H2D copy of one
    // sub-batch, the kernels of the next and the D2H copy of the previous one overlap
    hb_host::Lane lanes[hb_host::kLanes];
    // launch configuration, fixed at creation (configure_kernels): resident blocks per SM, decode layouts
    int sm_count = 148;
    int enc_blocks_per_sm[2] = {0, 0};  // encode_tiled_kernel<seg>
    int enc_slots_blocks_per_sm = 0;
    int str_blocks_per_sm[2] = {0, 0};  // str_bits_kernel, str_pack_kernel
    hb_host::DecLayout dec_layout[2];   // decode_batch_kernel<framed>
    hb_host::StreamLayout stream_layout;
    // staging for the host entry points
    GrowBuf s_in, s_in_off, s_out, s_out_off, s_caps, s_status, s_consumed, s_ovf_pattern, s_ovf_bits, s_left_bits,
        s_left_num;
    // HPACK string literals (hpack_literals.cuh): packed payloads between the framing and the codec, per-item plans
    GrowBuf hp_pay, hp_pay_off, hp_dec, hp_dec_off, hp_huff, hp_prefix, hp_lens, hp_pay_lens, hp_dec_status, hp_left_bits,
        hp_left_num, hp_status;
    hb_host::BlockBufs blk;
    uint64_t *h_scalar = nullptr;  // pinned
    // Calls enqueue on the caller's stream (device pointers) or on ctx->stream (host pointers) but share
    // ctx->scratch, the staging and the HPACK buffers. `scratch_free` is recorded after every such call; a call on
    // ANOTHER stream waits for it first, so two calls in flight on different streams never touch them at the same time.
    cudaEvent_t scratch_free = nullptr;
    cudaStream_t scratch_stream = nullptr;
    bool scratch_busy = false;
    // switches, read once at context creation (DESIGN.md 6b)
    bool force_generic = false, no_slots = false, no_strings = false, no_fused_stream = false;

    ~aws_huffman_batch_ctx() {
        if (h_scalar) cudaFreeHost(h_scalar);
        if (scratch_free) cudaEventDestroy(scratch_free);
        if (stream) cudaStreamDestroy(stream);
        if (d_enc) cudaFree(d_enc);
        if (d_lut) cudaFree(d_lut);
        if (d_lut2) cudaFree(d_lut2);
    }
};

namespace {

// Stream of a call on the context's shared buffers: the caller's, or the context's own (cuda_stream NULL, and every
// host-pointer call); ordered behind the previous call when that one ran on a different stream.
int call_begin(aws_huffman_batch_ctx *ctx, void *cuda_stream, cudaStream_t *st) {
    HB_CUDA_TRY(cudaSetDevice(ctx->device));
    *st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    if (ctx->scratch_busy && ctx->scratch_stream != *st) HB_CUDA_TRY(cudaStreamWaitEvent(*st, ctx->scratch_free, 0));
    return AWS_OP_SUCCESS;
}
int call_end(aws_huffman_batch_ctx *ctx, cudaStream_t st, int rc) {
    if (ctx->scratch_free && cudaEventRecord(ctx->scratch_free, st) == cudaSuccess) {
        ctx->scratch_stream = st;
        ctx->scratch_busy = true;
    } else {
        (void)cudaGetLastError();
    }
    return rc;
}

#ifndef HB_LUT_ROOT_BITS
#define HB_LUT_ROOT_BITS 12
#endif
constexpr uint32_t kLutRootBits = HB_LUT_ROOT_BITS;
constexpr uint32_t kLutSubBits = 8;
constexpr uint32_t kLutMaxSmemEntries = 8192;  // 32 KiB

int check_batch(const aws_huffman_batch *b) {
    if (!b) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (b->n == 0) return AWS_OP_SUCCESS;
    if (!b->in_offsets || !b->out_offsets) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

hb::BatchView make_view(const aws_huffman_batch *b) {
    hb::BatchView v{};
    v.n = b->n;
    v.in = b->in;
    v.in_offsets = b->in_offsets;
    v.out = b->out;
    v.out_capacity = b->out_capacity;
    v.out_offsets = b->out_offsets;
    v.out_caps = b->out_caps;
    v.out_lens = b->out_lens;
    v.status = b->status;
    v.consumed = b->consumed;
    v.overflow_pattern = b->overflow_pattern;
    v.overflow_num_bits = b->overflow_num_bits;
    v.leftover_working_bits = b->leftover_working_bits;
    v.leftover_num_bits = b->leftover_num_bits;
    return v;
}

// lens -> offsets on the device
int launch_scan(
    aws_huffman_batch_ctx *ctx, Scratch &sc, const uint64_t *lens, uint64_t *offsets, uint64_t n, cudaStream_t stream,
    const uint32_t *gate = nullptr, uint32_t slots_of = 0) {
    const uint64_t tiles = std::max<uint64_t>(1, (n + kScanTile - 1) / kScanTile);
    const size_t state_bytes = tiles * sizeof(uint64_t) + 256;
    HB_CUDA_TRY(sc.tile_state.reserve(state_bytes));
    HB_CUDA_TRY(cudaMemsetAsync(sc.tile_state.ptr, 0, state_bytes, stream));
    uint64_t *state = sc.tile_state.as<uint64_t>();
    uint32_t *ticket = reinterpret_cast<uint32_t *>(state + tiles);
    scan_lens_kernel<<<(unsigned)tiles, kScanThreads, 0, stream>>>(lens, offsets, n, state, ticket, gate, slots_of);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// Packed layout, many items, every symbol has a code: the tiled kernel with item-aligned thread ranges.
int encode_slots_on_device(
    aws_huffman_batch_ctx *ctx, Scratch &sc, const hb::BatchView &v, uint64_t total_in, cudaStream_t stream) {
    const uint64_t num_tiles_ub = (total_in / kEncSymsPerThread + v.n + kSlotsPerTile - 1) / kSlotsPerTile + 1;
    HB_CUDA_TRY(sc.slot_base.reserve((v.n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(sc.tile_first.reserve((num_tiles_ub + 1) * sizeof(EncSlotTile)));
    // slot_base = exclusive scan of the items' slot counts, straight from the offsets
    if (launch_scan(ctx, sc, v.in_offsets, sc.slot_base.as<uint64_t>(), v.n, stream, nullptr, kEncSymsPerThread)) return AWS_OP_ERR;
    slot_tile_index_kernel<<<(unsigned)((num_tiles_ub + 1 + 255) / 256), 256, 0, stream>>>(
        v.in_offsets, sc.slot_base.as<uint64_t>(), v.n, total_in, num_tiles_ub + 1, sc.tile_first.as<EncSlotTile>());
    ++ctx->launches;
    const size_t state_bytes = num_tiles_ub * sizeof(uint64_t) + 256;
    HB_CUDA_TRY(sc.tile_state.reserve(state_bytes));
    HB_CUDA_TRY(cudaMemsetAsync(sc.tile_state.ptr, 0, state_bytes, stream));
    EncSlotArgs a{};
    a.in = v.in;
    a.in_offsets = v.in_offsets;
    a.n = v.n;
    a.total_in = total_in;
    a.out = v.out;
    a.out_capacity = v.out_capacity;
    a.out_offsets = v.out_offsets;
    a.slot_base = sc.slot_base.as<uint64_t>();
    a.tiles = sc.tile_first.as<EncSlotTile>();
    a.tile_state = sc.tile_state.as<uint64_t>();
    a.ticket = reinterpret_cast<uint32_t *>(a.tile_state + num_tiles_ub);
    a.num_tiles_ub = (uint32_t)num_tiles_ub;
    a.eos_padding = ctx->tables.eos_padding;
    const unsigned grid = (unsigned)std::min<uint64_t>(num_tiles_ub, (uint64_t)ctx->sm_count * ctx->enc_slots_blocks_per_sm);
    encode_slots_kernel<<<grid, kEncBlock, kEncSlotSmemBytes, stream>>>(ctx->tables.enc, a);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

int encode_tiled_on_device(
    aws_huffman_batch_ctx *ctx, Scratch &sc, const hb::BatchView &v, uint64_t total_in, cudaStream_t stream,
    const uint32_t *gate = nullptr);

// Packed layout, many short strings, every symbol has a code: one thread per string (encode_strings.cuh).
int encode_strings_on_device(
    aws_huffman_batch_ctx *ctx, Scratch &sc, const hb::BatchView &v, uint64_t total_in, cudaStream_t stream) {
    const uint64_t scan_tiles = (v.n + kStrScanTile - 1) / kStrScanTile;
    const uint64_t bits_tiles = (total_in + kBitsTileBytes - 1) / kBitsTileBytes;
    const uint32_t phase = (uint32_t)(reinterpret_cast<uintptr_t>(v.out) & 15);
    // a symbol encodes to at most 4 bytes
    const uint64_t cap_tiles = (4 * total_in + v.n + phase) / kStrTileBytes + 4;
    HB_CUDA_TRY(sc.str_state.reserve(scan_tiles * sizeof(uint64_t) + 64));
    HB_CUDA_TRY(sc.str_ctl.reserve(kStrCtlWords * sizeof(uint32_t)));
    HB_CUDA_TRY(sc.str_tiles.reserve(cap_tiles * sizeof(uint32_t)));
    HB_CUDA_TRY(sc.str_bits.reserve((v.n + 8) * sizeof(uint32_t)));
    HB_CUDA_TRY(sc.str_bits_first.reserve((bits_tiles + 1) * sizeof(uint32_t)));
    StrArgs a{};
    a.in = v.in;
    a.in_offsets = v.in_offsets;
    a.n = v.n;
    a.total_in = total_in;
    a.out = v.out;
    a.out_capacity = v.out_capacity;
    a.out_offsets = v.out_offsets;
    a.tile_state = sc.str_state.as<uint64_t>();
    a.control = sc.str_ctl.as<uint32_t>();
    a.tile_first = sc.str_tiles.as<uint32_t>();
    a.num_measure_tiles = (uint32_t)scan_tiles;
    a.out_phase = phase;
    a.eos_padding = ctx->tables.eos_padding;
    StrPrepArgs p{};
    p.in_offsets = v.in_offsets;
    p.n = v.n;
    p.total_in = total_in;
    p.bits = sc.str_bits.as<uint32_t>();
    p.bits_tile_first = sc.str_bits_first.as<uint32_t>();
    p.tile_state = a.tile_state;
    p.control = a.control;
    p.tile_first = a.tile_first;
    p.num_bits_tiles = (uint32_t)bits_tiles;
    p.num_scan_tiles = (uint32_t)scan_tiles;
    StrBitsArgs m{};
    m.in = v.in;
    m.in_offsets = v.in_offsets;
    m.n = v.n;
    m.total_in = total_in;
    m.bits_tile_first = p.bits_tile_first;
    m.bits = p.bits;
    m.control = a.control;
    m.num_bits_tiles = (uint32_t)bits_tiles;
    const unsigned grid_prep = (unsigned)std::min<uint64_t>((v.n + 256) / 256, (uint64_t)ctx->sm_count * 16);
    str_prep_kernel<<<grid_prep, 256, 0, stream>>>(p);
    const unsigned grid_b = (unsigned)std::min<uint64_t>(std::max<uint64_t>(1, bits_tiles), (uint64_t)ctx->sm_count * ctx->str_blocks_per_sm[0]);
    str_bits_kernel<<<grid_b, kBitsThreads, 0, stream>>>(ctx->tables.enc, m);
    const unsigned grid_s = (unsigned)scan_tiles;
    str_scan_kernel<<<grid_s, kStrThreads, 0, stream>>>(p.bits, a);
    const unsigned grid_p = (unsigned)std::min<uint64_t>(cap_tiles, (uint64_t)ctx->sm_count * ctx->str_blocks_per_sm[1]);
    str_pack_kernel<<<grid_p, kStrThreads, kStrPackSmemBytes, stream>>>(ctx->tables.enc, a);
    ctx->launches += 4;
    HB_CUDA_TRY(cudaGetLastError());
    // strings this path does not take (very long ones): the tiled kernel redoes the batch, on the device's own flag
    return encode_tiled_on_device(ctx, sc, v, total_in, stream, a.control + kStrCtlFallback);
}

// Packed layout, every symbol has a code: the tiled symbol-parallel kernel.
int encode_tiled_on_device(
    aws_huffman_batch_ctx *ctx, Scratch &sc, const hb::BatchView &v, uint64_t total_in, cudaStream_t stream,
    const uint32_t *gate) {
    const uint64_t num_tiles = (total_in + kEncTile - 1) / kEncTile;
    const bool seg = v.n > 1;
    const size_t state_bytes = num_tiles * sizeof(uint64_t) + 256;
    HB_CUDA_TRY(sc.tile_state.reserve(state_bytes));
    HB_CUDA_TRY(cudaMemsetAsync(sc.tile_state.ptr, 0, state_bytes, stream));
    EncTiledArgs a{};
    a.in = v.in;
    a.in_offsets = v.in_offsets;
    a.n = v.n;
    a.total_in = total_in;
    a.out = v.out;
    a.out_capacity = v.out_capacity;
    a.out_offsets = v.out_offsets;
    a.tile_state = sc.tile_state.as<uint64_t>();
    a.ticket = reinterpret_cast<uint32_t *>(a.tile_state + num_tiles);
    a.num_tiles = (uint32_t)num_tiles;
    a.eos_padding = ctx->tables.eos_padding;
    a.gate = gate;
    if (seg) {
        HB_CUDA_TRY(sc.tile_first.reserve((num_tiles + 1) * sizeof(uint32_t)));
        a.tile_first = sc.tile_first.as<uint32_t>();
        tile_index_kernel<<<(unsigned)((num_tiles + 1 + 255) / 256), 256, 0, stream>>>(
            v.in_offsets, v.n, total_in, num_tiles, sc.tile_first.as<uint32_t>(), gate);
        ++ctx->launches;
    }
    const unsigned grid =
        (unsigned)std::min<uint64_t>(num_tiles, (uint64_t)ctx->sm_count * ctx->enc_blocks_per_sm[seg]);
    if (seg) encode_tiled_kernel<true><<<grid, kEncBlock, kEncSmemBytes, stream>>>(ctx->tables.enc, a);
    else encode_tiled_kernel<false><<<grid, kEncBlock, kEncSmemBytes, stream>>>(ctx->tables.enc, a);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

int encode_on_device(
    aws_huffman_batch_ctx *ctx, Scratch &sc, hb::BatchView v, uint64_t total_in, cudaStream_t stream) {
    if (v.n == 0) return AWS_OP_SUCCESS;
    const bool force_generic = ctx->force_generic;
    // (the tiled kernel's multiply-add accumulator needs 1 << len to fit a word: codes of up to 31 bits)
    if (!v.resume && !v.out_caps && !ctx->tables.has_unknown && ctx->tables.max_len <= 31 && total_in > 0 && v.n < 0xffffffffull &&
        (total_in + kEncTile - 1) / kEncTile < 0xffffffffull && !force_generic) {
        int rc;
        // many short strings: one thread per string
        if (v.n > 1 && total_in / v.n <= 2048 && (reinterpret_cast<uintptr_t>(v.in) & 15) == 0 &&
            (4 * total_in + v.n) / kStrTileBytes < 0xfffffff0ull && !ctx->no_strings)
            rc = encode_strings_on_device(ctx, sc, v, total_in, stream);
        // many items of some length: thread ranges aligned to the items
        else if (v.n > 1 && total_in / v.n >= 24 && total_in < (1ull << 31) && (reinterpret_cast<uintptr_t>(v.in) & 15) == 0 &&
                 !ctx->no_slots)
            rc = encode_slots_on_device(ctx, sc, v, total_in, stream);
        else
            rc = encode_tiled_on_device(ctx, sc, v, total_in, stream);
        if (rc) return AWS_OP_ERR;
        if (v.out_lens || v.status || v.consumed || v.overflow_pattern || v.overflow_num_bits) {
            fill_packed_meta_kernel<<<(unsigned)((v.n + 255) / 256), 256, 0, stream>>>(
                v.n, v.in_offsets, v.out_offsets, v.out_lens, v.status, v.consumed, v.overflow_pattern, v.overflow_num_bits);
            ++ctx->launches;
            HB_CUDA_TRY(cudaGetLastError());
        }
        return AWS_OP_SUCCESS;
    }
    if (!v.out_lens) {
        HB_CUDA_TRY(sc.lens.reserve(v.n * sizeof(uint64_t)));
        v.out_lens = sc.lens.as<uint64_t>();
    }
    const unsigned blocks = (unsigned)((v.n + kWarpsPerBlock - 1) / kWarpsPerBlock);
    if (!v.out_caps) {
        encode_items_warp_kernel<false><<<blocks, kWarpsPerBlock * 32, 0, stream>>>(ctx->tables, v);
        ++ctx->launches;
        HB_CUDA_TRY(cudaGetLastError());
        if (launch_scan(ctx, sc, v.out_lens, v.out_offsets, v.n, stream)) return AWS_OP_ERR;
    }
    encode_items_warp_kernel<true><<<blocks, kWarpsPerBlock * 32, 0, stream>>>(ctx->tables, v);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// Packed layout, many strings: fused count -> look-back -> write kernel (one thread per string).
int decode_batch_fast(
    aws_huffman_batch_ctx *ctx, Scratch &sc, const hb::BatchView &v, uint64_t total_in, cudaStream_t stream,
    bool framed = false) {
    DecBatchArgs a{};
    a.b = v;
    a.lut = ctx->tables.lut;
    a.lut2 = ctx->d_lut2;
    a.lut2_count = ctx->lut2_count;
    a.lut2_trap = ctx->lut2_trap;
    a.root_bits = ctx->tables.lut_root_bits;
    a.min_len = std::max<uint32_t>(1, ctx->tables.min_len);
    const hb_host::DecLayout &L = ctx->dec_layout[framed];
    const size_t stage_bytes = L.stage_bytes, rows_bytes = L.rows_bytes;
    const double expand = 8.0 / a.min_len;
    a.stage_words = (uint32_t)(stage_bytes / 4 - 2);
    a.rows_bytes = (uint32_t)rows_bytes;
    // strings per tile: as many as fit the stage and the row area at the batch's average length, with room to spare
    // for tiles above the average (a tile that does not fit takes the two-pass global route and every tile behind it
    // waits for its count)
    {
        const double avg = std::max(1.0, (double)total_in / (double)v.n);
        // (17 % to spare: on the benchmark's uniform 8..256 B strings a tile's bytes vary by 3.2 % (one sigma); with 12 %
        // two tiles in 4,500 overflowed, 20 % cost the ninth group of the tile)
        const double by_stage = (double)(stage_bytes - 64) / (1.17 * avg);
        const double by_rows = (double)rows_bytes / (1.17 * avg * expand + kDecRowSlack);
        const uint64_t fit = (uint64_t)std::max(32.0, std::min(by_stage, by_rows));
        // (in steps of 8 strings: the last group of a tile may be partly empty — it holds the tile's shortest strings —
        // and every string more per tile is decode-phase time shared by one more: 272 instead of 256 on the benchmark)
        a.items_per_tile = (uint32_t)std::min<uint64_t>(kDecItemsPerTile, std::max<uint64_t>(32, fit & ~uint64_t(7)));
    }
    const uint64_t num_tiles = (v.n + a.items_per_tile - 1) / a.items_per_tile;
    const size_t state_bytes = num_tiles * sizeof(uint64_t) + 256;
    HB_CUDA_TRY(sc.tile_state.reserve(state_bytes));
    HB_CUDA_TRY(cudaMemsetAsync(sc.tile_state.ptr, 0, state_bytes, stream));
    a.tile_state = sc.tile_state.as<uint64_t>();
    a.ticket = reinterpret_cast<uint32_t *>(a.tile_state + num_tiles);
    a.num_tiles = (uint32_t)num_tiles;
    const unsigned blocks = (unsigned)std::min<uint64_t>((num_tiles + kDecTeams - 1) / kDecTeams, (uint64_t)ctx->sm_count);
    if (framed) decode_batch_kernel<true><<<blocks, kDecTeams * kDecBlock, L.smem, stream>>>(a);
    else decode_batch_kernel<false><<<blocks, kDecTeams * kDecBlock, L.smem, stream>>>(a);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// Packed layout, one long stream: chunked speculative decode. The fused single-pass kernel does the
// work; the multi-kernel path behind it only runs (on the device's own decision, no host round trip)
// when the fused kernel raised its `fail` flag: a stream that does not self-synchronise, or that stops
// at an unknown symbol before its end.
int decode_stream_fast(
    aws_huffman_batch_ctx *ctx, Scratch &sc, const hb::BatchView &v, uint64_t len, cudaStream_t stream) {
    const uint64_t lead = reinterpret_cast<uintptr_t>(v.in) & 15;  // "aligned space" starts on a 16-byte boundary
    const uint64_t end_bit = (lead + len) * 8;
    const uint64_t num_chunks = (end_bit + kChunkBits - 1) / kChunkBits;
    HB_CUDA_TRY(sc.chunks.reserve(num_chunks * sizeof(uint64_t) + 64));
    HB_CUDA_TRY(sc.chunk_lens.reserve(num_chunks * sizeof(uint64_t)));
    HB_CUDA_TRY(sc.chunk_offsets.reserve((num_chunks + 1) * sizeof(uint64_t)));
    StreamArgs a{};
    a.in_aligned = v.in - lead;
    a.begin_bit = lead * 8;
    a.end_bit = end_bit;
    a.num_chunks = num_chunks;
    a.chunks = sc.chunks.as<uint64_t>();
    a.chunk_offsets = sc.chunk_offsets.as<uint64_t>();
    a.control = a.chunks + num_chunks;  // two words after the records
    a.lut = ctx->tables.lut;
    a.lut_count = ctx->tables.lut_count;
    a.root_bits = ctx->tables.lut_root_bits;
    const hb_host::StreamLayout &L = ctx->stream_layout;

    // ---- fused single pass ------------------------------------------------------------------------------------
    if (L.fused) {
        StreamFusedArgs f{};
        f.s = a;
        f.s.num_chunks = std::max<uint64_t>(1, (end_bit > 31 ? end_bit - 31 + kChunkBits - 1 : 0) / kChunkBits);
        f.b = v;
        f.num_tiles = (uint32_t)((f.s.num_chunks + kStreamThreads - 1) / kStreamThreads);
        f.row_words = L.row_words;
        f.lut2 = ctx->d_lut2;
        f.lut2_count = ctx->lut2_count;
        f.lut2_trap = ctx->lut2_trap;
        // [tile_state: num_tiles][tile_rec: num_tiles][ticket][fail]
        const size_t words = 2 * (size_t)f.num_tiles + 2;
        HB_CUDA_TRY(sc.fused.reserve(words * sizeof(uint64_t)));
        HB_CUDA_TRY(cudaMemsetAsync(sc.fused.ptr, 0, words * sizeof(uint64_t), stream));
        f.tile_state = sc.fused.as<uint64_t>();
        f.tile_rec = f.tile_state + f.num_tiles;
        f.ticket = reinterpret_cast<uint32_t *>(f.tile_rec + f.num_tiles);
        f.fail = f.ticket + 2;
        a.gate = f.fail;
        const unsigned blocks = (unsigned)std::min<uint64_t>((f.num_tiles + kStreamTeams - 1) / kStreamTeams, (uint64_t)ctx->sm_count);
        stream_fused_kernel<<<blocks, kStreamTeams * kStreamTeamThreads, L.fused_smem, stream>>>(f);
        stream_fused_verify_kernel<<<(unsigned)std::min<uint64_t>((f.num_tiles + 255) / 256, 1024), 256, 0, stream>>>(f);
        ctx->launches += 2;
        HB_CUDA_TRY(cudaGetLastError());
    }

    // ---- multi-kernel path (alone, or gated behind the fused kernel's fail flag) ----------------------------------
    HB_CUDA_TRY(cudaMemsetAsync(a.control, 0xff, 2 * sizeof(uint64_t), stream));
    // a gated launch that finds the flag clear costs a few microseconds: keep those grids small
    const uint64_t cap_wide = L.fused ? (uint64_t)ctx->sm_count * 4 : (uint64_t)ctx->sm_count * 12;
    const uint64_t cap_flat = L.fused ? (uint64_t)ctx->sm_count * 4 : (uint64_t)ctx->sm_count * 8;
    const unsigned wide = (unsigned)std::min<uint64_t>((num_chunks + kStreamThreads - 1) / kStreamThreads, cap_wide);
    const unsigned flat = (unsigned)std::min<uint64_t>((num_chunks + 255) / 256, cap_flat);
    stream_sync_kernel<<<wide, kStreamThreads, L.smem_staged, stream>>>(a);
    for (int round = 0; round < 2; ++round) stream_fix_kernel<<<wide, kStreamThreads, L.smem, stream>>>(a);
    stream_verify_kernel<<<flat, 256, 0, stream>>>(a);
    stream_repair_kernel<<<1, 32, L.smem, stream>>>(a);
    stream_counts_kernel<<<flat, 256, 0, stream>>>(a, sc.chunk_lens.as<uint64_t>());
    ctx->launches += 6;
    HB_CUDA_TRY(cudaGetLastError());
    if (launch_scan(ctx, sc, sc.chunk_lens.as<uint64_t>(), a.chunk_offsets, num_chunks, stream, a.gate)) return AWS_OP_ERR;
    stream_write_kernel<<<wide, kStreamThreads, L.smem_staged, stream>>>(a, v);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

constexpr uint64_t kStreamMinBytes = 64 * 1024;  // shorter single items go through the batch kernel

int decode_on_device(
    aws_huffman_batch_ctx *ctx, Scratch &sc, hb::BatchView v, uint64_t total_in, cudaStream_t stream) {
    if (v.n == 0) return AWS_OP_SUCCESS;
    const bool force_generic = ctx->force_generic;
    if (!v.resume && !v.out_caps && ctx->tables.lut_count <= kDecLutMaxSmem && !force_generic) {
        if (v.n == 1 && total_in >= kStreamMinBytes) return decode_stream_fast(ctx, sc, v, total_in, stream);
        return decode_batch_fast(ctx, sc, v, total_in, stream);
    }
    if (!v.out_lens) {
        HB_CUDA_TRY(sc.lens.reserve(v.n * sizeof(uint64_t)));
        v.out_lens = sc.lens.as<uint64_t>();
    }
    const unsigned threads = 256;
    const unsigned blocks = (unsigned)((v.n + threads - 1) / threads);
    const size_t smem = ctx->lut_smem_entries * sizeof(uint32_t);
    if (!v.out_caps) {
        decode_items_thread_kernel<false><<<blocks, threads, smem, stream>>>(ctx->tables, v, ctx->lut_smem_entries);
        ++ctx->launches;
        HB_CUDA_TRY(cudaGetLastError());
        if (launch_scan(ctx, sc, v.out_lens, v.out_offsets, v.n, stream)) return AWS_OP_ERR;
    }
    decode_items_thread_kernel<true><<<blocks, threads, smem, stream>>>(ctx->tables, v, ctx->lut_smem_entries);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

__global__ void rebase_offsets_kernel(const uint64_t *src, uint64_t count, uint64_t base, uint64_t *dst) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dst[i] = src[i] - base;
}

__global__ void add_base_kernel(uint64_t *offsets, uint64_t count, uint64_t base) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) offsets[i] += base;
}

// offsets[0..count) += base on the device (0 - b subtracts b: the sum wraps).
int add_base(aws_huffman_batch_ctx *ctx, uint64_t *offsets, uint64_t count, uint64_t base, cudaStream_t st) {
    if (base == 0 || count == 0) return AWS_OP_SUCCESS;
    add_base_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(offsets, count, base);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

int lane_prepare(Lane &lane) {
    if (lane.stream) return AWS_OP_SUCCESS;
    HB_CUDA_TRY(cudaStreamCreateWithFlags(&lane.stream, cudaStreamNonBlocking));
    HB_CUDA_TRY(cudaEventCreateWithFlags(&lane.kernels_done, cudaEventDisableTiming));
    HB_CUDA_TRY(cudaEventCreateWithFlags(&lane.retired, cudaEventDisableTiming));
    HB_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&lane.h_total), sizeof(uint64_t), cudaHostAllocDefault));
    return AWS_OP_SUCCESS;
}

constexpr uint64_t kPipelineMinBytes = 8ull << 20;   // below this one shot is as good
constexpr uint64_t kPipelineShardBytes = 12ull << 20;  // measured on PCIe Gen5 x16: 4 / 6 / 8 / 12 / 16 MiB: 53.2 / 57.0 / 58.3 / 60.4 / 59.6 GB/s
                                                       // end to end (round 1, slower kernels: 8 MiB)
// A sub-batch is retired (its D2H copies queued) one issue after it was issued, and its lane takes the next
// sub-batch kLanes issues after it took this one. A lane must not be re-used before its sub-batch was retired; with
// one lane more than that, re-using a lane never has to wait for a D2H copy that is still running, so uploads of
// later sub-batches and downloads of earlier ones stay concurrent.
constexpr size_t kRetireLag = 1;
static_assert(hb_host::kLanes >= kRetireLag + 2, "lanes must outnumber the issue-to-retire distance by two");

// Copies the per-item arrays of items [first, first + count) from the device view `v` into the caller's batch `b`.
// `v` holds an array exactly when the caller asked for it.
int copy_item_arrays_to_host(const aws_huffman_batch *b, const hb::BatchView &v, size_t first, size_t count, cudaStream_t st) {
    if (v.out_lens)
        HB_CUDA_TRY(cudaMemcpyAsync(b->out_lens + first, v.out_lens, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (v.status)
        HB_CUDA_TRY(cudaMemcpyAsync(b->status + first, v.status, count * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (v.consumed)
        HB_CUDA_TRY(cudaMemcpyAsync(b->consumed + first, v.consumed, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (v.overflow_pattern)
        HB_CUDA_TRY(cudaMemcpyAsync(
            b->overflow_pattern + first, v.overflow_pattern, count * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    if (v.overflow_num_bits)
        HB_CUDA_TRY(cudaMemcpyAsync(b->overflow_num_bits + first, v.overflow_num_bits, count, cudaMemcpyDeviceToHost, st));
    if (v.leftover_working_bits)
        HB_CUDA_TRY(cudaMemcpyAsync(
            b->leftover_working_bits + first, v.leftover_working_bits, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (v.leftover_num_bits)
        HB_CUDA_TRY(cudaMemcpyAsync(b->leftover_num_bits + first, v.leftover_num_bits, count, cudaMemcpyDeviceToHost, st));
    return AWS_OP_SUCCESS;
}

// Host-pointer staging: grows `buf` to `room` bytes, uploads `count` elements of `src` to it on `st` and sets `*dev`
// to the device copy (count 0: only the room, for an array the call writes).
template <typename T, typename D>
int stage_in(GrowBuf &buf, size_t room, const T *src, size_t count, cudaStream_t st, D **dev) {
    HB_CUDA_TRY(buf.reserve(room));
    if (count) HB_CUDA_TRY(cudaMemcpyAsync(buf.ptr, src, count * sizeof(T), cudaMemcpyHostToDevice, st));
    *dev = static_cast<D *>(buf.ptr);
    return AWS_OP_SUCCESS;
}

// The end of a host-pointer call with a packed result: offsets[0..count] (and status[0..count) when the caller asked
// for it) come down; then AWS_ERROR_SHORT_BUFFER when offsets[count] > capacity, else the payload of offsets[count]
// bytes is enqueued (d_out == NULL: there is none). The caller synchronises `st` after its last copy.
int finish_packed(cudaStream_t st, size_t count, const uint64_t *d_offsets, uint64_t *offsets, const void *d_out,
                  void *out, uint64_t capacity, const int32_t *d_status = nullptr, int32_t *status = nullptr) {
    HB_CUDA_TRY(cudaMemcpyAsync(offsets, d_offsets, (count + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (status && d_status) HB_CUDA_TRY(cudaMemcpyAsync(status, d_status, count * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    const uint64_t total = offsets[count];
    if (total > capacity) return aws_raise_error(AWS_ERROR_SHORT_BUFFER);
    if (d_out && total) HB_CUDA_TRY(cudaMemcpyAsync(out, d_out, total, cudaMemcpyDeviceToHost, st));
    return AWS_OP_SUCCESS;
}

// One value the host needs before it can go on (an output size): copied down and waited for.
int read_back(const uint64_t *d_value, uint64_t *value, cudaStream_t st) {
    HB_CUDA_TRY(cudaMemcpyAsync(value, d_value, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    return AWS_OP_SUCCESS;
}

// The end of a host-pointer call for one slice of its items (all of them, or one shard of a multi call) whose packed
// output starts at `base` in the caller's arrays: the slice's `count` offsets, and the closing one when the slice is
// the last, are rebased on the device and come down to `offsets`, with status when the caller asked for it. Then
// AWS_ERROR_SHORT_BUFFER when the whole call's output `total` is over `capacity` (offsets and status are complete),
// else the slice's `size` payload octets go to out + base (d_out == NULL: there is none). The caller synchronises
// `st` after its last copy.
int finish_slice(aws_huffman_batch_ctx *ctx, cudaStream_t st, size_t count, bool last, uint64_t *d_offsets, uint64_t *offsets,
                 uint64_t base, const void *d_out, void *out, uint64_t size, uint64_t total, uint64_t capacity,
                 const int32_t *d_status = nullptr, int32_t *status = nullptr) {
    const size_t entries = count + (last ? 1 : 0);
    if (add_base(ctx, d_offsets, entries, base, st)) return AWS_OP_ERR;
    if (entries) HB_CUDA_TRY(cudaMemcpyAsync(offsets, d_offsets, entries * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (status && d_status && count)
        HB_CUDA_TRY(cudaMemcpyAsync(status, d_status, count * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (total > capacity) {
        HB_CUDA_TRY(cudaStreamSynchronize(st));
        return aws_raise_error(AWS_ERROR_SHORT_BUFFER);
    }
    if (d_out && size) HB_CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t *>(out) + base, d_out, size, cudaMemcpyDeviceToHost, st));
    return AWS_OP_SUCCESS;
}

// Packed layout with many items: the batch is cut into sub-batches (contiguous item ranges balanced by
// bytes) that flow through kLanes lanes, so the host->device copy of one sub-batch, the kernels of the
// next and the device->host copy of the previous one run at the same time. Sub-batches are ordinary
// independent batches on the device; their packed offsets are rebased on the host at the end
// (the same concatenation step as multi-GPU sharding). Only the lanes' own buffers are used, none of the
// context's shared ones, so this path needs no call_begin / call_end.
int run_host_batch_pipelined(aws_huffman_batch_ctx *ctx, const aws_huffman_batch *b, bool encode) {
    HB_CUDA_TRY(cudaSetDevice(ctx->device));
    const size_t n = b->n;
    const uint64_t total_in = b->in_offsets[n];
    size_t shards = (size_t)std::min<uint64_t>(256, std::max<uint64_t>(2, total_in / kPipelineShardBytes));
    shards = std::min(shards, n);
    std::vector<size_t> begin(shards + 1);
    if (aws_huffman_batch_plan_shards(b->in_offsets, n, shards, begin.data())) return AWS_OP_ERR;
    // One item larger than a sub-batch's share makes several byte targets fall inside it: plan_shards then
    // returns empty ranges. An empty sub-batch has nothing to issue or retire (its out_offsets[0] would never
    // be written on the device), so the ranges are compacted first.
    begin.erase(std::unique(begin.begin(), begin.end()), begin.end());
    shards = begin.size() - 1;
    // (cutting the first and last sub-batches smaller, to shorten pipeline fill and drain, was measured: no
    // effect — 59.5 vs 60.2 GB/s end to end)
    std::vector<hb::BatchView> views(shards);  // sub-batch j's arrays on the device, read back by retire(j)

    for (Lane &lane : ctx->lanes)
        if (lane_prepare(lane)) return AWS_OP_ERR;

    const uint32_t max_len = std::max<uint32_t>(1, ctx->tables.max_len);
    const uint32_t min_len = std::max<uint32_t>(1, ctx->tables.min_len);
    uint64_t base_out = 0;
    bool overflow = false;

    auto issue = [&](size_t j) -> int {
        Lane &lane = ctx->lanes[j % hb_host::kLanes];
        if (lane.in_flight) {
            HB_CUDA_TRY(cudaEventSynchronize(lane.retired));
            lane.in_flight = false;
        }
        const size_t a = begin[j], nj = begin[j + 1] - a;
        const uint64_t in0 = b->in_offsets[a], bytes_in = b->in_offsets[a + nj] - in0;
        const uint64_t room = encode ? bytes_in * ((max_len + 7) / 8) + 64 : (bytes_in * 8) / min_len + 64;
        HB_CUDA_TRY(lane.in.reserve(bytes_in + 64));
        HB_CUDA_TRY(lane.in_off.reserve((nj + 1) * sizeof(uint64_t)));
        HB_CUDA_TRY(lane.out.reserve(room + 64));
        HB_CUDA_TRY(lane.out_off.reserve((nj + 1) * sizeof(uint64_t)));
        if (b->out_lens) HB_CUDA_TRY(lane.lens.reserve(nj * sizeof(uint64_t)));
        if (b->status) HB_CUDA_TRY(lane.status.reserve(nj * sizeof(int32_t)));
        if (b->consumed) HB_CUDA_TRY(lane.consumed.reserve(nj * sizeof(uint64_t)));
        if (encode ? b->overflow_pattern != nullptr : false) HB_CUDA_TRY(lane.aux32.reserve(nj * sizeof(uint32_t)));
        if (encode ? b->overflow_num_bits != nullptr : b->leftover_num_bits != nullptr) HB_CUDA_TRY(lane.aux8.reserve(nj));
        if (!encode && b->leftover_working_bits) HB_CUDA_TRY(lane.aux64.reserve(nj * sizeof(uint64_t)));

        // the sub-batch's slice of the offsets goes up with it and is rebased in place on the device
        HB_CUDA_TRY(cudaMemcpyAsync(
            lane.in_off.ptr, b->in_offsets + a, (nj + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, lane.stream));
        if (bytes_in)
            HB_CUDA_TRY(cudaMemcpyAsync(lane.in.ptr, b->in + in0, bytes_in, cudaMemcpyHostToDevice, lane.stream));
        rebase_offsets_kernel<<<(unsigned)((nj + 1 + 255) / 256), 256, 0, lane.stream>>>(
            lane.in_off.as<uint64_t>(), nj + 1, in0, lane.in_off.as<uint64_t>());
        ++ctx->launches;
        hb::BatchView &v = views[j];
        v.n = nj;
        v.in = lane.in.as<uint8_t>();
        v.in_offsets = lane.in_off.as<uint64_t>();
        v.out = lane.out.as<uint8_t>();
        v.out_capacity = room;
        v.out_offsets = lane.out_off.as<uint64_t>();
        v.out_lens = b->out_lens ? lane.lens.as<uint64_t>() : nullptr;
        v.status = b->status ? lane.status.as<int32_t>() : nullptr;
        v.consumed = b->consumed ? lane.consumed.as<uint64_t>() : nullptr;
        if (encode) {
            v.overflow_pattern = b->overflow_pattern ? lane.aux32.as<uint32_t>() : nullptr;
            v.overflow_num_bits = b->overflow_num_bits ? lane.aux8.as<uint8_t>() : nullptr;
        } else {
            v.leftover_working_bits = b->leftover_working_bits ? lane.aux64.as<uint64_t>() : nullptr;
            v.leftover_num_bits = b->leftover_num_bits ? lane.aux8.as<uint8_t>() : nullptr;
        }
        if ((encode ? encode_on_device(ctx, lane.scratch, v, bytes_in, lane.stream)
                    : decode_on_device(ctx, lane.scratch, v, bytes_in, lane.stream)) != AWS_OP_SUCCESS)
            return AWS_OP_ERR;
        HB_CUDA_TRY(cudaMemcpyAsync(
            lane.h_total, lane.out_off.as<uint64_t>() + nj, sizeof(uint64_t), cudaMemcpyDeviceToHost, lane.stream));
        HB_CUDA_TRY(cudaEventRecord(lane.kernels_done, lane.stream));
        lane.in_flight = true;
        return AWS_OP_SUCCESS;
    };

    auto retire = [&](size_t j) -> int {
        Lane &lane = ctx->lanes[j % hb_host::kLanes];
        const size_t a = begin[j], nj = begin[j + 1] - a;
        HB_CUDA_TRY(cudaEventSynchronize(lane.kernels_done));
        const uint64_t total = *lane.h_total;
        cudaStream_t st = lane.stream;
        if (base_out + total > b->out_capacity) overflow = true;
        if (!overflow && total)
            HB_CUDA_TRY(cudaMemcpyAsync(b->out + base_out, lane.out.ptr, total, cudaMemcpyDeviceToHost, st));
        if (base_out) {
            // the concatenation step: shard-local packed offsets -> global, before they leave the device
            add_base_kernel<<<(unsigned)((nj + 255) / 256), 256, 0, st>>>(lane.out_off.as<uint64_t>(), nj, base_out);
            ++ctx->launches;
        }
        HB_CUDA_TRY(cudaMemcpyAsync(b->out_offsets + a, lane.out_off.ptr, nj * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        if (copy_item_arrays_to_host(b, views[j], a, nj, st)) return AWS_OP_ERR;
        HB_CUDA_TRY(cudaEventRecord(lane.retired, st));
        base_out += total;
        return AWS_OP_SUCCESS;
    };

    // On an error no copy into the caller's buffers may still be running when the call returns.
    auto drain = [&]() {
        for (Lane &lane : ctx->lanes) {
            if (lane.stream) (void)cudaStreamSynchronize(lane.stream);
            lane.in_flight = false;
        }
        (void)cudaGetLastError();
    };
    for (size_t j = 0; j < shards + kRetireLag; ++j) {
        if ((j < shards && issue(j)) || (j >= kRetireLag && retire(j - kRetireLag))) {
            const int err = aws_last_error();
            drain();
            return aws_raise_error(err ? err : AWS_ERROR_COMPRESSION_DEVICE_FAILURE);
        }
    }
    for (Lane &lane : ctx->lanes) {
        if (lane.in_flight) HB_CUDA_TRY(cudaEventSynchronize(lane.retired));
        lane.in_flight = false;
    }
    b->out_offsets[n] = base_out;
    if (overflow) return aws_raise_error(AWS_ERROR_SHORT_BUFFER);
    return AWS_OP_SUCCESS;
}

int check_resume(const aws_huffman_batch *b, bool encode) {
    // the state arrays are inputs as well as outputs
    if (b && b->n &&
        (encode ? (!b->overflow_pattern || !b->overflow_num_bits) : (!b->leftover_working_bits || !b->leftover_num_bits)))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

// One host-pointer call through the context's staging: stage in, run, stage out.
int run_host_batch_staged(aws_huffman_batch_ctx *ctx, const aws_huffman_batch *b, bool encode, bool resume, cudaStream_t st) {
    const size_t n = b->n;
    const uint64_t total_in = b->in_offsets[n];
    const bool slotted = b->out_caps != nullptr;
    const size_t up = resume ? n : 0;  // (the resume state goes up; otherwise those arrays are outputs only)
    hb::BatchView v{};
    v.resume = resume;
    v.n = n;
    v.out_capacity = b->out_capacity;
    // (slotted: bytes the codec does not touch must come back unchanged, so the output goes up too)
    if (stage_in(ctx->s_in, total_in + 16, b->in, total_in, st, &v.in) ||
        stage_in(ctx->s_in_off, (n + 1) * sizeof(uint64_t), b->in_offsets, n + 1, st, &v.in_offsets) ||
        stage_in(ctx->s_out, b->out_capacity + 16, b->out, slotted ? b->out_capacity : 0, st, &v.out) ||
        stage_in(ctx->s_out_off, (n + 1) * sizeof(uint64_t), b->out_offsets, slotted ? n : 0, st, &v.out_offsets) ||
        (slotted && stage_in(ctx->s_caps, n * sizeof(uint64_t), b->out_caps, n, st, &v.out_caps)) ||
        (b->status && stage_in(ctx->s_status, n * sizeof(int32_t), b->status, 0, st, &v.status)) ||
        (b->consumed && stage_in(ctx->s_consumed, n * sizeof(uint64_t), b->consumed, 0, st, &v.consumed)))
        return AWS_OP_ERR;
    if (encode) {
        if ((b->overflow_pattern &&
             stage_in(ctx->s_ovf_pattern, n * sizeof(uint32_t), b->overflow_pattern, up, st, &v.overflow_pattern)) ||
            (b->overflow_num_bits && stage_in(ctx->s_ovf_bits, n, b->overflow_num_bits, up, st, &v.overflow_num_bits)))
            return AWS_OP_ERR;
    } else if ((b->leftover_working_bits && stage_in(ctx->s_left_bits, n * sizeof(uint64_t), b->leftover_working_bits, up,
                                                     st, &v.leftover_working_bits)) ||
               (b->leftover_num_bits && stage_in(ctx->s_left_num, n, b->leftover_num_bits, up, st, &v.leftover_num_bits))) {
        return AWS_OP_ERR;
    }
    HB_CUDA_TRY(ctx->scratch.lens.reserve(n * sizeof(uint64_t)));
    v.out_lens = b->out_lens ? ctx->scratch.lens.as<uint64_t>() : nullptr;

    if ((encode ? encode_on_device(ctx, ctx->scratch, v, total_in, st)
                : decode_on_device(ctx, ctx->scratch, v, total_in, st)) != AWS_OP_SUCCESS)
        return AWS_OP_ERR;

    if (copy_item_arrays_to_host(b, v, 0, n, st)) return AWS_OP_ERR;
    if (slotted) {
        if (b->out_capacity) HB_CUDA_TRY(cudaMemcpyAsync(b->out, v.out, b->out_capacity, cudaMemcpyDeviceToHost, st));
    } else if (finish_packed(st, n, v.out_offsets, b->out_offsets, v.out, b->out, b->out_capacity)) {
        return AWS_OP_ERR;
    }
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    return AWS_OP_SUCCESS;
}

// Host-pointer entry point shared by encode and decode.
int run_host_batch(aws_huffman_batch_ctx *ctx, const aws_huffman_batch *b, bool encode, bool resume = false) {
    if (!ctx) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (check_batch(b)) return AWS_OP_ERR;
    if (resume && check_resume(b, encode)) return AWS_OP_ERR;
    const size_t n = b->n;
    if (n == 0) {
        if (!b->out_caps && b->out_offsets) b->out_offsets[0] = 0;
        return AWS_OP_SUCCESS;
    }
    const uint64_t total_in = b->in_offsets[n];
    if ((total_in && !b->in) || (b->out_capacity && !b->out)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    // (payloads are always staged through device memory, pinned caller buffers too: kernels that read and write pinned
    // host memory over PCIe measured slower end to end than the copy engines, DESIGN.md 6)
    if (!resume && !b->out_caps && n >= 2 && total_in >= kPipelineMinBytes) return run_host_batch_pipelined(ctx, b, encode);
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, run_host_batch_staged(ctx, b, encode, resume, st));
}

// An empty packed batch on the device: its whole result is out_offsets[0] = 0 (NULL: nothing to write).
int write_empty_packed(uint64_t *out_offsets, cudaStream_t st) {
    if (out_offsets) HB_CUDA_TRY(cudaMemsetAsync(out_offsets, 0, sizeof(uint64_t), st));
    return AWS_OP_SUCCESS;
}

// Device-pointer entry point shared by encode and decode.
int run_device_batch(aws_huffman_batch_ctx *ctx, const aws_huffman_batch *b, void *cuda_stream, bool encode, bool resume) {
    if (!ctx) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (check_batch(b) || (resume && check_resume(b, encode))) return AWS_OP_ERR;
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    if (b->n == 0) return call_end(ctx, st, b->out_caps ? AWS_OP_SUCCESS : write_empty_packed(b->out_offsets, st));
    hb::BatchView v = make_view(b);
    v.resume = resume;
    return call_end(ctx, st, encode ? encode_on_device(ctx, ctx->scratch, v, b->in_size, st)
                                    : decode_on_device(ctx, ctx->scratch, v, b->in_size, st));
}

// ---------------------------------------------------------------------------------------------
// HPACK string literals (SURVEY.md 8f.1). Device pointers in, device pointers out.
// ---------------------------------------------------------------------------------------------
int hpack_encode_on_device(
    aws_huffman_batch_ctx *ctx, uint64_t n, const uint8_t *raw, const uint64_t *raw_off, uint64_t total_in, uint32_t mode,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_off, cudaStream_t st) {
    if (n == 0) return AWS_OP_SUCCESS;
    const unsigned flat = (unsigned)((n + 255) / 256), warps = (unsigned)((n + 255) / 256);  // (move kernels: 32 items per warp)
    HB_CUDA_TRY(ctx->hp_huff.reserve(n));
    HB_CUDA_TRY(ctx->hp_lens.reserve(n * sizeof(uint64_t)));
    const uint8_t *pay = nullptr;
    const uint64_t *pay_off = nullptr;
    if (mode != hb::kHpackNever) {
        const uint64_t cap = total_in * ((std::max<uint32_t>(1, ctx->tables.max_len) + 7) / 8) + 64;
        HB_CUDA_TRY(ctx->hp_pay.reserve(cap + 64));
        HB_CUDA_TRY(ctx->hp_pay_off.reserve((n + 1) * sizeof(uint64_t)));
        hb::BatchView v{};
        v.n = n;
        v.in = raw;
        v.in_offsets = raw_off;
        v.out = ctx->hp_pay.as<uint8_t>();
        v.out_capacity = cap;
        v.out_offsets = ctx->hp_pay_off.as<uint64_t>();
        if (encode_on_device(ctx, ctx->scratch, v, total_in, st)) return AWS_OP_ERR;
        pay = ctx->hp_pay.as<uint8_t>();
        pay_off = ctx->hp_pay_off.as<uint64_t>();
    }
    hb::hpack_plan_kernel<<<flat, 256, 0, st>>>(n, raw_off, pay_off, mode, ctx->hp_huff.as<uint8_t>(), ctx->hp_lens.as<uint64_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, ctx->hp_lens.as<uint64_t>(), out_off, n, st)) return AWS_OP_ERR;
    hb::hpack_frame_kernel<<<warps, 256, 0, st>>>(n, raw, raw_off, pay, pay_off, ctx->hp_huff.as<uint8_t>(), out, out_capacity, out_off);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

int hpack_decode_on_device(
    aws_huffman_batch_ctx *ctx, uint64_t n, const uint8_t *in, const uint64_t *in_off, uint64_t total_in, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_off, int32_t *status, cudaStream_t st) {
    if (n == 0) return AWS_OP_SUCCESS;
    // (the one-kernel route copies raw literals into rows sized 8 len / min_len: a table whose shortest code is longer
    // than a byte — not HPACK's — takes the multi-pass route)
    // (AWS_HUFFMAN_HPACK_PASSES is read per call, DESIGN.md 6b)
    if (n > 1 && ctx->tables.lut_count <= kDecLutMaxSmem && ctx->tables.min_len <= 8 && !ctx->force_generic &&
        !getenv("AWS_HUFFMAN_HPACK_PASSES")) {
        // one kernel: the batch decoder parses the literals in its string table, copies raw payloads, applies
        // the padding rule to what it leaves over and writes strings, offsets and status itself
        hb::BatchView v{};
        v.n = n;
        v.in = in;
        v.in_offsets = in_off;
        v.out = out;
        v.out_capacity = out_capacity;
        v.out_offsets = out_off;
        if (!status) {
            HB_CUDA_TRY(ctx->hp_status.reserve(n * sizeof(int32_t)));
            status = ctx->hp_status.as<int32_t>();
        }
        v.status = status;
        return decode_batch_fast(ctx, ctx->scratch, v, total_in, st, true);
    }
    // one long literal (chunked stream kernels) or a table too large for shared memory: framing passes around the codec
    const unsigned flat = (unsigned)((n + 255) / 256), warps = (unsigned)((n + 255) / 256);  // (move kernels: 32 items per warp)
    const uint32_t min_len = std::max<uint32_t>(1, ctx->tables.min_len);
    const uint64_t dec_cap = total_in * 8 / min_len + 64;
    HB_CUDA_TRY(ctx->hp_huff.reserve(n));
    HB_CUDA_TRY(ctx->hp_prefix.reserve(n));
    HB_CUDA_TRY(ctx->hp_lens.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(ctx->hp_pay_lens.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(ctx->hp_pay.reserve(total_in + 64));
    HB_CUDA_TRY(ctx->hp_pay_off.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(ctx->hp_dec.reserve(dec_cap + 64));
    HB_CUDA_TRY(ctx->hp_dec_off.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(ctx->hp_dec_status.reserve(n * sizeof(int32_t)));
    HB_CUDA_TRY(ctx->hp_left_bits.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(ctx->hp_left_num.reserve(n));
    if (!status) {
        HB_CUDA_TRY(ctx->hp_status.reserve(n * sizeof(int32_t)));
        status = ctx->hp_status.as<int32_t>();
    }
    uint8_t *huff = ctx->hp_huff.as<uint8_t>(), *prefix = ctx->hp_prefix.as<uint8_t>();
    uint64_t *pay_lens = ctx->hp_pay_lens.as<uint64_t>(), *lens = ctx->hp_lens.as<uint64_t>();
    uint64_t *pay_off = ctx->hp_pay_off.as<uint64_t>(), *dec_off = ctx->hp_dec_off.as<uint64_t>();

    // 1. parse the literals; 2. the Huffman payloads, packed
    hb::hpack_parse_kernel<<<flat, 256, 0, st>>>(n, in, in_off, huff, prefix, pay_lens, lens, status);
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, lens, pay_off, n, st)) return AWS_OP_ERR;
    hb::hpack_move_kernel<<<warps, 256, 0, st>>>(
        n, in, in_off, prefix, pay_lens, nullptr, nullptr, huff, false, true, status, ctx->hp_pay.as<uint8_t>(), total_in, pay_off);
    ++ctx->launches;
    // 3. decode them (the single-stream kernels size themselves from the payload length: needed on the host for n == 1)
    uint64_t pay_total = total_in;
    if (n == 1) {
        if (!ctx->h_scalar) HB_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_scalar), sizeof(uint64_t), cudaHostAllocDefault));
        HB_CUDA_TRY(cudaMemcpyAsync(ctx->h_scalar, pay_off + 1, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        HB_CUDA_TRY(cudaStreamSynchronize(st));
        pay_total = *ctx->h_scalar;
    }
    hb::BatchView v{};
    v.n = n;
    v.in = ctx->hp_pay.as<uint8_t>();
    v.in_offsets = pay_off;
    v.out = ctx->hp_dec.as<uint8_t>();
    v.out_capacity = dec_cap;
    v.out_offsets = dec_off;
    v.status = ctx->hp_dec_status.as<int32_t>();
    v.leftover_working_bits = ctx->hp_left_bits.as<uint64_t>();
    v.leftover_num_bits = ctx->hp_left_num.as<uint8_t>();
    if (decode_on_device(ctx, ctx->scratch, v, pay_total, st)) return AWS_OP_ERR;
    // 4. padding rule, final lengths; 5. the strings, packed
    hb::hpack_finish_kernel<<<flat, 256, 0, st>>>(
        n, huff, pay_lens, dec_off, v.status, v.leftover_working_bits, v.leftover_num_bits, status, lens);
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, lens, out_off, n, st)) return AWS_OP_ERR;
    hb::hpack_move_kernel<<<warps, 256, 0, st>>>(
        n, in, in_off, prefix, pay_lens, ctx->hp_dec.as<uint8_t>(), dec_off, huff, true, false, status, out, out_capacity, out_off);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// Host pointers, run on the device: the n items of in_off[0..n] (offsets into the caller's `in`) are staged from
// octet in_base on, their offsets rebased to it, and framed or decoded into the context's staging, out_capacity
// octets at most; *size receives the output size. hpack_run_finish then writes them into the caller's arrays.
int hpack_run_slice(
    aws_huffman_batch_ctx *ctx, bool encode, size_t n, const uint8_t *in, const uint64_t *in_off, uint64_t in_base,
    uint32_t mode, uint64_t out_capacity, uint64_t *size, cudaStream_t st) {
    const uint64_t total_in = in_off[n] - in_base;
    const uint8_t *d_in = nullptr;
    uint64_t *d_in_off = nullptr;
    if (stage_in(ctx->s_in, total_in + 16, in + in_base, total_in, st, &d_in) ||
        stage_in(ctx->s_in_off, (n + 1) * sizeof(uint64_t), in_off, n + 1, st, &d_in_off) ||
        add_base(ctx, d_in_off, n + 1, 0 - in_base, st))
        return AWS_OP_ERR;
    HB_CUDA_TRY(ctx->s_out.reserve(out_capacity + 16));
    HB_CUDA_TRY(ctx->s_out_off.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(ctx->s_status.reserve(n * sizeof(int32_t)));
    uint8_t *d_out = ctx->s_out.as<uint8_t>();
    uint64_t *d_out_off = ctx->s_out_off.as<uint64_t>();
    int32_t *d_status = ctx->s_status.as<int32_t>();
    if (encode ? hpack_encode_on_device(ctx, n, d_in, d_in_off, total_in, mode, d_out, out_capacity, d_out_off, st)
               : hpack_decode_on_device(ctx, n, d_in, d_in_off, total_in, d_out, out_capacity, d_out_off, d_status, st))
        return AWS_OP_ERR;
    return read_back(d_out_off + n, size, st);
}

// Host pointers, finish into place: the items hpack_run_slice ran are the caller's from out_off / status on (the
// closing offset too when `last`), their `size` octets go to out + base; `total`, the output size of the whole call,
// decides AWS_ERROR_SHORT_BUFFER.
int hpack_run_finish(
    aws_huffman_batch_ctx *ctx, bool encode, size_t n, bool last, uint64_t base, uint64_t size, uint64_t total, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_off, int32_t *status, cudaStream_t st) {
    if (finish_slice(ctx, st, n, last, ctx->s_out_off.as<uint64_t>(), out_off, base, ctx->s_out.ptr, out, size, total,
                     out_capacity, encode ? nullptr : ctx->s_status.as<int32_t>(), status))
        return AWS_OP_ERR;
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    return AWS_OP_SUCCESS;
}

// Host pointers: run on the device, then finish at base 0.
int hpack_run_staged(
    aws_huffman_batch_ctx *ctx, bool encode, size_t n, const uint8_t *in, const uint64_t *in_off, uint32_t mode, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_off, int32_t *status, cudaStream_t st) {
    uint64_t size = 0;
    if (hpack_run_slice(ctx, encode, n, in, in_off, 0, mode, out_capacity, &size, st)) return AWS_OP_ERR;
    return hpack_run_finish(ctx, encode, n, true, 0, size, size, out, out_capacity, out_off, status, st);
}

// Arguments of the host-pointer literal calls; a call with no items is answered here (*done).
int hpack_host_args(size_t n, const uint8_t *in, const uint64_t *in_off, const uint8_t *out, uint64_t out_capacity,
                    uint64_t *out_off, bool *done) {
    *done = false;
    if (n && (!in_off || !out_off)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (n == 0) {
        if (out_off) out_off[0] = 0;
        *done = true;
        return AWS_OP_SUCCESS;
    }
    if ((in_off[n] && !in) || (out_capacity && !out)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

int hpack_run_host(
    aws_huffman_batch_ctx *ctx, bool encode, size_t n, const uint8_t *in, const uint64_t *in_off, uint32_t mode, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_off, int32_t *status) {
    bool done;
    if (!ctx) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (hpack_host_args(n, in, in_off, out, out_capacity, out_off, &done) || done) return done ? AWS_OP_SUCCESS : AWS_OP_ERR;
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, hpack_run_staged(ctx, encode, n, in, in_off, mode, out, out_capacity, out_off, status, st));
}

// ---------------------------------------------------------------------------------------------
// HPACK header blocks (hpack_blocks.cuh) over the literal layer above. Device pointers in, device pointers out.
// ---------------------------------------------------------------------------------------------
// Device pointers of an aws_hpack_header_lists (decode side).
struct BlockLists {
    uint64_t *field_offsets;
    uint64_t field_capacity;
    uint8_t *kind;
    uint64_t *index;
    uint8_t *strings;
    uint64_t strings_capacity;
    uint64_t *string_offsets;
};

inline unsigned grid_of(uint64_t items, uint64_t per_block) { return (unsigned)std::max<uint64_t>(1, (items + per_block - 1) / per_block); }

// stage: `o` holds host pointers' shapes only; the per-field outputs go to context staging sized from the totals
// (the host entry point copies them back).
int hpack_blocks_decode_on_device(
    aws_huffman_batch_ctx *ctx, uint64_t n, const uint8_t *in, const uint64_t *in_off, BlockLists o, int32_t *status,
    bool stage, cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    if (n == 0) {
        HB_CUDA_TRY(cudaMemsetAsync(o.field_offsets, 0, sizeof(uint64_t), st));
        if (o.string_offsets && !stage) HB_CUDA_TRY(cudaMemsetAsync(o.string_offsets, 0, sizeof(uint64_t), st));
        return AWS_OP_SUCCESS;
    }
    const unsigned flat = grid_of(n, 256);
    HB_CUDA_TRY(B.num_fields.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.num_lits.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_bytes.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.out_fields.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.struct_status.reserve(n * sizeof(int32_t)));
    HB_CUDA_TRY(B.field_base.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_base.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_byte_base.reserve((n + 1) * sizeof(uint64_t)));
    if (!status) {
        HB_CUDA_TRY(B.status.reserve(n * sizeof(int32_t)));
        status = B.status.as<int32_t>();
    }
    if (!B.h_totals) HB_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&B.h_totals), 3 * sizeof(uint64_t), cudaHostAllocDefault));
    uint64_t *field_base = B.field_base.as<uint64_t>(), *lit_base = B.lit_base.as<uint64_t>();
    uint64_t *lit_byte_base = B.lit_byte_base.as<uint64_t>();

    // 1. structure, counts; 2. their bases, and the totals the later launches are sized from
    hb::hpack_block_scan_kernel<<<flat, 256, 0, st>>>(
        n, in, in_off, B.num_fields.as<uint64_t>(), B.num_lits.as<uint64_t>(), B.lit_bytes.as<uint64_t>(), B.struct_status.as<int32_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.num_fields.as<uint64_t>(), field_base, n, st)) return AWS_OP_ERR;
    if (launch_scan(ctx, ctx->scratch, B.num_lits.as<uint64_t>(), lit_base, n, st)) return AWS_OP_ERR;
    if (launch_scan(ctx, ctx->scratch, B.lit_bytes.as<uint64_t>(), lit_byte_base, n, st)) return AWS_OP_ERR;
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 0, field_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 1, lit_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 2, lit_byte_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    const uint64_t parsed = B.h_totals[0], num_lits = B.h_totals[1], lit_total = B.h_totals[2];
    const uint64_t kept = std::min(parsed, o.field_capacity);  // field slots that can be written
    const uint32_t min_len = std::max<uint32_t>(1, ctx->tables.min_len);
    const uint64_t dec_cap = lit_total * 8 / min_len + 64;
    if (stage) {
        // (a field's strings are its decoded literals or at most 28 octets of Appendix A)
        o.strings_capacity = std::min(o.strings_capacity, dec_cap + 28 * kept);
        HB_CUDA_TRY(B.s_kind.reserve(kept + 1));
        HB_CUDA_TRY(B.s_index.reserve((kept + 1) * sizeof(uint64_t)));
        HB_CUDA_TRY(B.s_string_offsets.reserve((2 * kept + 1) * sizeof(uint64_t)));
        HB_CUDA_TRY(ctx->s_out.reserve(o.strings_capacity + 16));
        o.kind = B.s_kind.as<uint8_t>();
        o.index = B.s_index.as<uint64_t>();
        o.string_offsets = B.s_string_offsets.as<uint64_t>();
        o.strings = ctx->s_out.as<uint8_t>();
    }
    HB_CUDA_TRY(B.f_kind.reserve(parsed + 1));
    HB_CUDA_TRY(B.f_index.reserve((parsed + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.f_block.reserve((parsed + 1) * sizeof(uint32_t)));
    HB_CUDA_TRY(B.f_lits.reserve((2 * parsed + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_src.reserve((num_lits + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_offsets.reserve((num_lits + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_status.reserve((num_lits + 1) * sizeof(int32_t)));
    HB_CUDA_TRY(B.dec_offsets.reserve((num_lits + 1) * sizeof(uint64_t)));
    uint8_t *f_kind = B.f_kind.as<uint8_t>();
    uint64_t *f_index = B.f_index.as<uint64_t>(), *f_lits = B.f_lits.as<uint64_t>();
    uint32_t *f_block = B.f_block.as<uint32_t>();
    uint64_t *dec_offsets = B.dec_offsets.as<uint64_t>();
    int32_t *lit_status = B.lit_status.as<int32_t>();

    // 3. field records and literal spans in parsed order; 4. the literals, packed; 5. decoded by the literal path
    if (parsed || num_lits) {
        hb::hpack_block_split_kernel<<<flat, 256, 0, st>>>(
            n, in, in_off, field_base, lit_base, lit_byte_base, f_kind, f_index, f_block, f_lits, B.lit_src.as<uint64_t>(),
            B.lit_offsets.as<uint64_t>());
        ++ctx->launches;
    }
    if (num_lits) {
        HB_CUDA_TRY(B.lits.reserve(lit_total + 64));
        HB_CUDA_TRY(B.dec.reserve(dec_cap + 64));
        hb::hpack_lit_gather_kernel<<<grid_of(num_lits, 256), 256, 0, st>>>(
            num_lits, in, B.lit_src.as<uint64_t>(), B.lit_offsets.as<uint64_t>(), B.lits.as<uint8_t>());
        ++ctx->launches;
        if (hpack_decode_on_device(ctx, num_lits, B.lits.as<uint8_t>(), B.lit_offsets.as<uint64_t>(), lit_total,
                                   B.dec.as<uint8_t>(), dec_cap, dec_offsets, lit_status, st))
            return AWS_OP_ERR;
    }
    // 6. final status per block, field offsets; 7. records, string lengths, string offsets, strings
    hb::hpack_block_finish_kernel<<<flat, 256, 0, st>>>(
        n, lit_base, lit_status, B.struct_status.as<int32_t>(), B.num_fields.as<uint64_t>(), status, B.out_fields.as<uint64_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.out_fields.as<uint64_t>(), o.field_offsets, n, st)) return AWS_OP_ERR;
    if (!kept) {
        HB_CUDA_TRY(cudaMemsetAsync(o.string_offsets, 0, sizeof(uint64_t), st));
        HB_CUDA_TRY(cudaGetLastError());
        return AWS_OP_SUCCESS;
    }
    HB_CUDA_TRY(B.str_lens.reserve(2 * kept * sizeof(uint64_t)));
    HB_CUDA_TRY(cudaMemsetAsync(B.str_lens.ptr, 0, 2 * kept * sizeof(uint64_t), st));
    const uint8_t *dec = B.dec.as<uint8_t>();
    hb::hpack_field_records_kernel<hb::HpackFieldStrings><<<grid_of(parsed, 256), 256, 0, st>>>(
        parsed, f_kind, f_index, f_block, f_lits, field_base, status, o.field_offsets, o.field_capacity, dec, dec_offsets,
        o.kind, o.index, B.str_lens.as<uint64_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.str_lens.as<uint64_t>(), o.string_offsets, 2 * kept, st)) return AWS_OP_ERR;
    hb::hpack_compose_kernel<hb::HpackFieldStrings><<<grid_of(2 * parsed, 256), 256, 0, st>>>(
        parsed, f_kind, f_index, f_block, f_lits, field_base, status, o.field_offsets, o.field_capacity, dec, dec_offsets,
        o.strings, o.strings_capacity, o.string_offsets);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// field_kind == NULL: every field is AUTO (aws_hpack_header_block_encode_batch); else the caller's records, with
// the per-block status (optional) of aws_hpack_header_block_encode_records_batch.
int hpack_blocks_encode_on_device(
    aws_huffman_batch_ctx *ctx, uint64_t n, const uint64_t *field_offsets, uint64_t num_fields, const uint8_t *never_indexed,
    const uint8_t *field_kind, const uint64_t *field_index, const uint8_t *strings, const uint64_t *string_offsets,
    uint64_t strings_size, uint32_t mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status,
    cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    if (n == 0 || num_fields == 0) {
        HB_CUDA_TRY(cudaMemsetAsync(out_offsets, 0, (n + 1) * sizeof(uint64_t), st));
        if (status && n) HB_CUDA_TRY(cudaMemsetAsync(status, 0, n * sizeof(int32_t), st));
        return AWS_OP_SUCCESS;
    }
    const uint64_t F = num_fields;
    // framed names and values: raw or Huffman, whichever `mode` picks, behind a prefix of at most 10 octets
    const uint64_t expand = mode == hb::kHpackAlways ? (std::max<uint32_t>(1, ctx->tables.max_len) + 7) / 8 : 1;
    const uint64_t framed_cap = strings_size * expand + 2 * F * 10 + 64;
    HB_CUDA_TRY(B.framed.reserve(framed_cap + 64));
    HB_CUDA_TRY(B.framed_offsets.reserve((2 * F + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.plan.reserve(F));
    HB_CUDA_TRY(B.plan_index.reserve(F * sizeof(uint64_t)));
    HB_CUDA_TRY(B.field_lens.reserve(F * sizeof(uint64_t)));
    HB_CUDA_TRY(B.field_pos.reserve((F + 1) * sizeof(uint64_t)));
    const uint64_t *framed_offsets = B.framed_offsets.as<uint64_t>();
    uint64_t *field_pos = B.field_pos.as<uint64_t>();

    // 1. every name and value framed (indexed names too: simpler than a compacted batch); 2. representation and size
    // per field, and for records the block rules; 3. wire positions of fields and blocks; 4. prefixes and literals
    if (hpack_encode_on_device(ctx, 2 * F, strings, string_offsets, strings_size, mode, B.framed.as<uint8_t>(), framed_cap,
                               B.framed_offsets.as<uint64_t>(), st))
        return AWS_OP_ERR;
    hb::hpack_field_plan_kernel<<<grid_of(F, 256), 256, 0, st>>>(
        F, strings, string_offsets, never_indexed, field_kind, field_index, framed_offsets, B.plan.as<uint8_t>(),
        B.plan_index.as<uint64_t>(), B.field_lens.as<uint64_t>());
    ++ctx->launches;
    if (field_kind) {
        hb::hpack_block_check_kernel<<<grid_of(n, 256), 256, 0, st>>>(
            n, field_offsets, B.plan.as<uint8_t>(), B.field_lens.as<uint64_t>(), status);
        ++ctx->launches;
    }
    if (launch_scan(ctx, ctx->scratch, B.field_lens.as<uint64_t>(), field_pos, F, st)) return AWS_OP_ERR;
    hb::hpack_block_offsets_kernel<<<grid_of(n + 1, 256), 256, 0, st>>>(n, field_offsets, field_pos, out_offsets);
    ++ctx->launches;
    hb::hpack_field_emit_kernel<<<grid_of(F, 256), 256, 0, st>>>(
        F, B.plan.as<uint8_t>(), B.plan_index.as<uint64_t>(), B.framed.as<uint8_t>(), framed_offsets, field_pos, out,
        out_capacity);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

int check_block_lists(const aws_hpack_header_lists *l, bool decode) {
    if (!l || (l->n && !l->field_offsets) || !l->string_offsets || l->n > 0xffffffffull)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (decode && ((l->field_capacity && (!l->field_kind || !l->field_index)) || (l->strings_capacity && !l->strings)))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

// Offsets from the caller's memory, read before any kernel trusts them: a decreasing pair would send a walk or a
// copy outside the arrays.
bool offsets_sorted(const uint64_t *offsets, uint64_t count) {
    for (uint64_t i = 1; i < count; ++i)
        if (offsets[i] < offsets[i - 1]) return false;
    return true;
}

BlockLists block_lists(const aws_hpack_header_lists *l) {
    return BlockLists{l->field_offsets, l->field_capacity, l->field_kind, l->field_index, l->strings, l->strings_capacity,
                      l->string_offsets};
}

// Host pointers, run on the device (the way hpack_run_slice does): the n blocks of in_off[0..n] are staged from octet
// in_base on and decoded into the context's staging, within the capacities given; size[0] receives their fields and,
// when those fit field_capacity, size[1] their string octets.
int hpack_blocks_decode_slice(
    aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_off, uint64_t in_base,
    uint64_t field_capacity, uint64_t strings_capacity, uint64_t size[2], cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    const uint64_t total_in = in_off[n] - in_base;
    const uint8_t *d_in = nullptr;
    uint64_t *d_in_off = nullptr;
    BlockLists o{nullptr, field_capacity, nullptr, nullptr, nullptr, strings_capacity, nullptr};
    if (stage_in(ctx->s_in, total_in + 16, in + in_base, total_in, st, &d_in) ||
        stage_in(ctx->s_in_off, (n + 1) * sizeof(uint64_t), in_off, n + 1, st, &d_in_off) ||
        add_base(ctx, d_in_off, n + 1, 0 - in_base, st))
        return AWS_OP_ERR;
    HB_CUDA_TRY(B.s_field_offsets.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(ctx->s_status.reserve(n * sizeof(int32_t)));
    o.field_offsets = B.s_field_offsets.as<uint64_t>();
    if (hpack_blocks_decode_on_device(ctx, n, d_in, d_in_off, o, ctx->s_status.as<int32_t>(), true, st) ||
        read_back(o.field_offsets + n, &size[0], st))
        return AWS_OP_ERR;
    size[1] = 0;  // (string offsets exist for the fields that fit)
    return size[0] <= field_capacity ? read_back(B.s_string_offsets.as<uint64_t>() + 2 * size[0], &size[1], st) : AWS_OP_SUCCESS;
}

// Host pointers, finish into place: the blocks hpack_blocks_decode_slice ran are the caller's from block `first` on,
// their fields from field base[0] on and their string octets from base[1] on; `total` (fields, string octets) of the
// whole call decides AWS_ERROR_SHORT_BUFFER.
int hpack_blocks_decode_finish(
    aws_huffman_batch_ctx *ctx, size_t first, size_t n, bool last, const uint64_t base[2], const uint64_t size[2],
    const uint64_t total[2], aws_hpack_header_lists *out, int32_t *status, cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    const uint64_t fields = size[0];
    // field records (no payload of their own here), then the strings behind them
    if (finish_slice(ctx, st, n, last, B.s_field_offsets.as<uint64_t>(), out->field_offsets + first, base[0], nullptr, nullptr,
                     0, total[0], out->field_capacity, ctx->s_status.as<int32_t>(), status ? status + first : nullptr) ||
        finish_slice(ctx, st, 2 * fields, last, B.s_string_offsets.as<uint64_t>(), out->string_offsets + 2 * base[0], base[1],
                     ctx->s_out.ptr, out->strings, size[1], total[1], out->strings_capacity))
        return AWS_OP_ERR;
    if (fields) {
        HB_CUDA_TRY(cudaMemcpyAsync(out->field_kind + base[0], B.s_kind.ptr, fields, cudaMemcpyDeviceToHost, st));
        HB_CUDA_TRY(cudaMemcpyAsync(out->field_index + base[0], B.s_index.ptr, fields * sizeof(uint64_t),
                                    cudaMemcpyDeviceToHost, st));
    }
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    return AWS_OP_SUCCESS;
}

// Host pointers: run on the device, then finish at base 0.
int hpack_blocks_decode_staged(
    aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_off, aws_hpack_header_lists *out,
    int32_t *status, cudaStream_t st) {
    const uint64_t base[2] = {0, 0};
    uint64_t size[2];
    if (hpack_blocks_decode_slice(ctx, n, in, in_off, 0, out->field_capacity, out->strings_capacity, size, st))
        return AWS_OP_ERR;
    return hpack_blocks_decode_finish(ctx, 0, n, true, base, size, size, out, status, st);
}

// Arguments of the host-pointer decode calls; a call with no blocks is answered here (*done).
int hpack_blocks_decode_args(size_t n, const uint8_t *in, const uint64_t *in_off, aws_hpack_header_lists *out, bool *done) {
    *done = false;
    if ((n && !in_off) || check_block_lists(out, true) || out->n != n) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (n == 0) {
        out->field_offsets[0] = 0;
        out->string_offsets[0] = 0;
        *done = true;
        return AWS_OP_SUCCESS;
    }
    if ((in_off[n] && !in) || !offsets_sorted(in_off, n + 1)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

int hpack_blocks_decode_host(
    aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_off, aws_hpack_header_lists *out,
    int32_t *status) {
    bool done;
    if (!ctx) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (hpack_blocks_decode_args(n, in, in_off, out, &done) || done) return done ? AWS_OP_SUCCESS : AWS_OP_ERR;
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, hpack_blocks_decode_staged(ctx, n, in, in_off, out, status, st));
}

// Host pointers, run on the device: lists [first, first + n) of `in` are staged, their field and string offsets
// rebased to their first field and first string octet, and encoded into the context's staging, out_capacity octets at
// most; *size receives the output size. records: field_kind and field_index are read
// (aws_hpack_header_block_encode_records_batch) and a status per list is written to the staging.
int hpack_blocks_encode_slice(
    aws_huffman_batch_ctx *ctx, const aws_hpack_header_lists *in, size_t first, size_t n, bool records, uint32_t mode,
    uint64_t out_capacity, uint64_t *size, cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    const uint64_t f0 = in->field_offsets[first], F = in->field_offsets[first + n] - f0;
    const uint64_t s0 = in->string_offsets[2 * f0], S = in->string_offsets[2 * (f0 + F)] - s0;
    uint64_t *d_field_offsets = nullptr, *d_string_offsets = nullptr;
    const uint8_t *d_strings = nullptr, *never = nullptr, *kind = nullptr;
    const uint64_t *index = nullptr;
    int32_t *d_status = nullptr;
    if (records) {
        HB_CUDA_TRY(ctx->s_status.reserve(n * sizeof(int32_t)));
        d_status = ctx->s_status.as<int32_t>();
    }
    if (stage_in(B.s_field_offsets, (n + 1) * sizeof(uint64_t), in->field_offsets + first, n + 1, st, &d_field_offsets) ||
        add_base(ctx, d_field_offsets, n + 1, 0 - f0, st) ||
        stage_in(ctx->s_in, S + 16, in->strings + s0, S, st, &d_strings) ||
        stage_in(ctx->s_in_off, (2 * F + 1) * sizeof(uint64_t), in->string_offsets + 2 * f0, 2 * F + 1, st, &d_string_offsets) ||
        add_base(ctx, d_string_offsets, 2 * F + 1, 0 - s0, st) ||
        (in->never_indexed && F && stage_in(B.s_never, F, in->never_indexed + f0, F, st, &never)) ||
        (records && (stage_in(B.s_kind, F + 1, in->field_kind + f0, F, st, &kind) ||
                     stage_in(B.s_index, (F + 1) * sizeof(uint64_t), in->field_index + f0, F, st, &index))))
        return AWS_OP_ERR;
    HB_CUDA_TRY(ctx->s_out.reserve(out_capacity + 16));
    HB_CUDA_TRY(ctx->s_out_off.reserve((n + 1) * sizeof(uint64_t)));
    if (hpack_blocks_encode_on_device(ctx, n, d_field_offsets, F, never, kind, index, d_strings, d_string_offsets, S, mode,
                                      ctx->s_out.as<uint8_t>(), out_capacity, ctx->s_out_off.as<uint64_t>(), d_status, st))
        return AWS_OP_ERR;
    return read_back(ctx->s_out_off.as<uint64_t>() + n, size, st);
}

// Host pointers, finish into place: the lists hpack_blocks_encode_slice ran are the caller's from list `first` on,
// their `size` octets go to out + base; `total`, the output size of the whole call, decides AWS_ERROR_SHORT_BUFFER.
int hpack_blocks_encode_finish(
    aws_huffman_batch_ctx *ctx, size_t first, size_t n, bool last, bool records, uint64_t base, uint64_t size, uint64_t total,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_off, int32_t *status, cudaStream_t st) {
    if (finish_slice(ctx, st, n, last, ctx->s_out_off.as<uint64_t>(), out_off + first, base, ctx->s_out.ptr, out, size, total,
                     out_capacity, records ? ctx->s_status.as<int32_t>() : nullptr, status ? status + first : nullptr))
        return AWS_OP_ERR;
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    return AWS_OP_SUCCESS;
}

// Host pointers: run on the device, then finish at base 0.
int hpack_blocks_encode_staged(
    aws_huffman_batch_ctx *ctx, const aws_hpack_header_lists *in, bool records, uint32_t mode, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_off, int32_t *status, cudaStream_t st) {
    uint64_t size = 0;
    if (hpack_blocks_encode_slice(ctx, in, 0, in->n, records, mode, out_capacity, &size, st)) return AWS_OP_ERR;
    return hpack_blocks_encode_finish(ctx, 0, in->n, true, records, 0, size, size, out, out_capacity, out_off, status, st);
}

// Arguments of the host-pointer encode calls; a call with no lists is answered here (*done).
int hpack_blocks_encode_args(const aws_hpack_header_lists *in, bool records, const uint8_t *out, uint64_t out_capacity,
                             uint64_t *out_off, bool *done) {
    *done = false;
    if (check_block_lists(in, false) || !out_off || (out_capacity && !out) || (records && (!in->field_kind || !in->field_index)))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    const uint64_t n = in->n;
    if (n == 0) {
        out_off[0] = 0;
        *done = true;
        return AWS_OP_SUCCESS;
    }
    // (fields are numbered from 0 and every one is encoded: lists start at field 0, strings at octet 0)
    if (in->field_offsets[0] != 0 || !offsets_sorted(in->field_offsets, n + 1)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    const uint64_t F = in->field_offsets[n];
    if (in->string_offsets[0] != 0 || !offsets_sorted(in->string_offsets, 2 * F + 1))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (in->string_offsets[2 * F] && !in->strings) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

int hpack_blocks_encode_host(
    aws_huffman_batch_ctx *ctx, const aws_hpack_header_lists *in, bool records, uint32_t mode, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_off, int32_t *status) {
    bool done;
    if (!ctx) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (hpack_blocks_encode_args(in, records, out, out_capacity, out_off, &done) || done)
        return done ? AWS_OP_SUCCESS : AWS_OP_ERR;
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, hpack_blocks_encode_staged(ctx, in, records, mode, out, out_capacity, out_off, status, st));
}

// ---------------------------------------------------------------------------------------------
// QPACK field sections (qpack_sections.cuh) over the same literal layer, the same buffers and the same passes as the
// HPACK header blocks above. Device pointers in, device pointers out.
// ---------------------------------------------------------------------------------------------
// stage: `o` holds the prefix arrays and field_offsets (context staging) and the capacities; the per-field outputs go
// to context staging sized from the totals (the host entry point copies them back).
int qpack_sections_decode_on_device(
    aws_huffman_batch_ctx *ctx, uint64_t n, const uint8_t *in, const uint64_t *in_off, aws_qpack_field_sections o,
    int32_t *status, bool stage, cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    if (n == 0) {
        HB_CUDA_TRY(cudaMemsetAsync(o.field_offsets, 0, sizeof(uint64_t), st));
        if (o.string_offsets && !stage) HB_CUDA_TRY(cudaMemsetAsync(o.string_offsets, 0, sizeof(uint64_t), st));
        return AWS_OP_SUCCESS;
    }
    const unsigned flat = grid_of(n, 256);
    HB_CUDA_TRY(B.num_fields.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.num_lits.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_bytes.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.out_fields.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.struct_status.reserve(n * sizeof(int32_t)));
    HB_CUDA_TRY(B.field_base.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_base.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_byte_base.reserve((n + 1) * sizeof(uint64_t)));
    if (!status) {
        HB_CUDA_TRY(B.status.reserve(n * sizeof(int32_t)));
        status = B.status.as<int32_t>();
    }
    if (!B.h_totals) HB_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&B.h_totals), 3 * sizeof(uint64_t), cudaHostAllocDefault));
    uint64_t *field_base = B.field_base.as<uint64_t>(), *lit_base = B.lit_base.as<uint64_t>();
    uint64_t *lit_byte_base = B.lit_byte_base.as<uint64_t>();

    // 1. structure, counts; 2. their bases, and the totals the later launches are sized from
    hb::qpack_section_scan_kernel<<<flat, 256, 0, st>>>(
        n, in, in_off, B.num_fields.as<uint64_t>(), B.num_lits.as<uint64_t>(), B.lit_bytes.as<uint64_t>(), B.struct_status.as<int32_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.num_fields.as<uint64_t>(), field_base, n, st)) return AWS_OP_ERR;
    if (launch_scan(ctx, ctx->scratch, B.num_lits.as<uint64_t>(), lit_base, n, st)) return AWS_OP_ERR;
    if (launch_scan(ctx, ctx->scratch, B.lit_bytes.as<uint64_t>(), lit_byte_base, n, st)) return AWS_OP_ERR;
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 0, field_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 1, lit_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 2, lit_byte_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    const uint64_t parsed = B.h_totals[0], num_lits = B.h_totals[1], lit_total = B.h_totals[2];
    const uint64_t kept = std::min(parsed, o.field_capacity);  // field slots that can be written
    const uint32_t min_len = std::max<uint32_t>(1, ctx->tables.min_len);
    const uint64_t dec_cap = lit_total * 8 / min_len + 64;
    if (stage) {
        // (a field's strings are its decoded literals or at most 69 octets of Appendix A)
        o.strings_capacity = std::min(o.strings_capacity, dec_cap + 69 * kept);
        HB_CUDA_TRY(B.s_kind.reserve(kept + 1));
        HB_CUDA_TRY(B.s_index.reserve((kept + 1) * sizeof(uint64_t)));
        HB_CUDA_TRY(B.s_never.reserve(kept + 1));
        HB_CUDA_TRY(B.s_string_offsets.reserve((2 * kept + 1) * sizeof(uint64_t)));
        HB_CUDA_TRY(ctx->s_out.reserve(o.strings_capacity + 16));
        o.field_kind = B.s_kind.as<uint8_t>();
        o.field_index = B.s_index.as<uint64_t>();
        o.never_indexed = B.s_never.as<uint8_t>();
        o.string_offsets = B.s_string_offsets.as<uint64_t>();
        o.strings = ctx->s_out.as<uint8_t>();
    }
    HB_CUDA_TRY(B.f_kind.reserve(parsed + 1));
    HB_CUDA_TRY(B.f_index.reserve((parsed + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.f_block.reserve((parsed + 1) * sizeof(uint32_t)));
    HB_CUDA_TRY(B.f_lits.reserve((2 * parsed + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_src.reserve((num_lits + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_len.reserve((num_lits + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_offsets.reserve((num_lits + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_status.reserve((num_lits + 1) * sizeof(int32_t)));
    HB_CUDA_TRY(B.dec_offsets.reserve((num_lits + 1) * sizeof(uint64_t)));
    uint8_t *f_kind = B.f_kind.as<uint8_t>();
    uint64_t *f_index = B.f_index.as<uint64_t>(), *f_lits = B.f_lits.as<uint64_t>();
    uint32_t *f_block = B.f_block.as<uint32_t>();
    uint64_t *dec_offsets = B.dec_offsets.as<uint64_t>();
    int32_t *lit_status = B.lit_status.as<int32_t>();

    // 3. field records and literals in parsed order; 4. the literals, packed and re-framed as RFC 7541 5.2 literals;
    // 5. decoded by the literal path
    if (parsed || num_lits) {
        hb::qpack_section_split_kernel<<<flat, 256, 0, st>>>(
            n, in, in_off, field_base, lit_base, lit_byte_base, f_kind, f_index, f_block, f_lits, B.lit_src.as<uint64_t>(),
            B.lit_len.as<uint64_t>(), B.lit_offsets.as<uint64_t>());
        ++ctx->launches;
    }
    if (num_lits) {
        HB_CUDA_TRY(B.lits.reserve(lit_total + 64));
        HB_CUDA_TRY(B.dec.reserve(dec_cap + 64));
        hb::qpack_lit_gather_kernel<<<grid_of(num_lits, 256), 256, 0, st>>>(
            num_lits, in, B.lit_src.as<uint64_t>(), B.lit_len.as<uint64_t>(), B.lit_offsets.as<uint64_t>(), B.lits.as<uint8_t>());
        ++ctx->launches;
        if (hpack_decode_on_device(ctx, num_lits, B.lits.as<uint8_t>(), B.lit_offsets.as<uint64_t>(), lit_total,
                                   B.dec.as<uint8_t>(), dec_cap, dec_offsets, lit_status, st))
            return AWS_OP_ERR;
    }
    // 6. final status per section, its prefix, field offsets; 7. records, string lengths, string offsets, strings
    hb::hpack_block_finish_kernel<<<flat, 256, 0, st>>>(
        n, lit_base, lit_status, B.struct_status.as<int32_t>(), B.num_fields.as<uint64_t>(), status, B.out_fields.as<uint64_t>());
    ++ctx->launches;
    hb::qpack_section_prefix_kernel<<<flat, 256, 0, st>>>(n, in, in_off, status, o.encoded_insert_count, o.base_sign,
                                                           o.delta_base);
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.out_fields.as<uint64_t>(), o.field_offsets, n, st)) return AWS_OP_ERR;
    if (!kept) {
        HB_CUDA_TRY(cudaMemsetAsync(o.string_offsets, 0, sizeof(uint64_t), st));
        HB_CUDA_TRY(cudaGetLastError());
        return AWS_OP_SUCCESS;
    }
    HB_CUDA_TRY(B.str_lens.reserve(2 * kept * sizeof(uint64_t)));
    HB_CUDA_TRY(cudaMemsetAsync(B.str_lens.ptr, 0, 2 * kept * sizeof(uint64_t), st));
    const uint8_t *dec = B.dec.as<uint8_t>();
    hb::qpack_field_records_kernel<<<grid_of(parsed, 256), 256, 0, st>>>(
        parsed, f_kind, f_index, f_block, f_lits, field_base, status, o.field_offsets, o.field_capacity, dec, dec_offsets,
        o.field_kind, o.field_index, o.never_indexed, B.str_lens.as<uint64_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.str_lens.as<uint64_t>(), o.string_offsets, 2 * kept, st)) return AWS_OP_ERR;
    hb::hpack_compose_kernel<hb::QpackFieldStrings><<<grid_of(2 * parsed, 256), 256, 0, st>>>(
        parsed, f_kind, f_index, f_block, f_lits, field_base, status, o.field_offsets, o.field_capacity, dec, dec_offsets,
        o.strings, o.strings_capacity, o.string_offsets);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// eic == NULL: stateless (aws_qpack_field_section_encode_batch: field_kind and field_index are NULL too); else the
// caller's records and prefixes, with the per-section status (optional) of aws_qpack_field_section_encode_records_batch.
int qpack_sections_encode_on_device(
    aws_huffman_batch_ctx *ctx, uint64_t n, const uint64_t *field_offsets, uint64_t num_fields, const uint8_t *never_indexed,
    const uint8_t *field_kind, const uint64_t *field_index, const uint64_t *eic, const uint8_t *sign, const uint64_t *delta,
    const uint8_t *strings, const uint64_t *string_offsets, uint64_t strings_size, uint32_t mode, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_offsets, int32_t *status, cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    if (n == 0) {
        HB_CUDA_TRY(cudaMemsetAsync(out_offsets, 0, sizeof(uint64_t), st));
        return AWS_OP_SUCCESS;
    }
    const uint64_t F = num_fields;
    HB_CUDA_TRY(B.sec_lens.reserve(n * sizeof(uint64_t)));
    const uint64_t *framed_offsets = nullptr;
    uint64_t *field_pos = nullptr;
    // 1. every name and value framed; 2. line and size per field (sections without fields skip both)
    if (F) {
        const uint64_t expand = mode == hb::kHpackAlways ? (std::max<uint32_t>(1, ctx->tables.max_len) + 7) / 8 : 1;
        const uint64_t framed_cap = strings_size * expand + 2 * F * 10 + 64;
        HB_CUDA_TRY(B.framed.reserve(framed_cap + 64));
        HB_CUDA_TRY(B.framed_offsets.reserve((2 * F + 1) * sizeof(uint64_t)));
        HB_CUDA_TRY(B.plan.reserve(F));
        HB_CUDA_TRY(B.plan_index.reserve(F * sizeof(uint64_t)));
        HB_CUDA_TRY(B.field_lens.reserve(F * sizeof(uint64_t)));
        HB_CUDA_TRY(B.field_pos.reserve((F + 1) * sizeof(uint64_t)));
        framed_offsets = B.framed_offsets.as<uint64_t>();
        field_pos = B.field_pos.as<uint64_t>();
        if (hpack_encode_on_device(ctx, 2 * F, strings, string_offsets, strings_size, mode, B.framed.as<uint8_t>(), framed_cap,
                                   B.framed_offsets.as<uint64_t>(), st))
            return AWS_OP_ERR;
        hb::qpack_field_plan_kernel<<<grid_of(F, 256), 256, 0, st>>>(
            F, strings, string_offsets, never_indexed, field_kind, field_index, B.framed.as<uint8_t>(), framed_offsets,
            B.plan.as<uint8_t>(), B.plan_index.as<uint64_t>(), B.field_lens.as<uint64_t>());
        ++ctx->launches;
    }
    // 3. the section rules and sizes (prefix included); 4. wire positions of sections and fields; 5. prefixes, and
    // the fields placed behind them; 6. the lines
    hb::qpack_section_size_kernel<<<grid_of(n, 256), 256, 0, st>>>(
        n, field_offsets, eic, sign, delta, B.plan.as<uint8_t>(), B.field_lens.as<uint64_t>(), status, B.sec_lens.as<uint64_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.sec_lens.as<uint64_t>(), out_offsets, n, st)) return AWS_OP_ERR;
    if (F && launch_scan(ctx, ctx->scratch, B.field_lens.as<uint64_t>(), field_pos, F, st)) return AWS_OP_ERR;
    hb::qpack_section_place_kernel<<<grid_of(n, 256), 256, 0, st>>>(n, field_offsets, eic, sign, delta, out_offsets,
                                                                     field_pos, out, out_capacity);
    ++ctx->launches;
    if (F) {
        hb::qpack_field_emit_kernel<hb::QpackFieldLines><<<grid_of(F, 256), 256, 0, st>>>(
            F, B.plan.as<uint8_t>(), B.plan_index.as<uint64_t>(), B.framed.as<uint8_t>(), framed_offsets, field_pos, out,
            out_capacity);
        ++ctx->launches;
    }
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// The argument rules of check_block_lists, and the prefix arrays: written by a decode, read by a records encode.
int check_section_lists(const aws_qpack_field_sections *l, bool decode, bool records) {
    if (!l || (l->n && !l->field_offsets) || !l->string_offsets || l->n > 0xffffffffull)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (decode && ((l->field_capacity && (!l->field_kind || !l->field_index || !l->never_indexed)) ||
                   (l->strings_capacity && !l->strings)))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if ((decode || records) && l->n && (!l->encoded_insert_count || !l->base_sign || !l->delta_base))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (records && (!l->field_kind || !l->field_index)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

// Host pointers, run on the device (the way hpack_blocks_decode_slice does): the n sections are staged and decoded into
// the context's staging, within the capacities given; size[0] receives their fields and, when those fit
// field_capacity, size[1] their string octets.
int qpack_sections_decode_slice(
    aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_off, uint64_t field_capacity,
    uint64_t strings_capacity, uint64_t size[2], cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    const uint64_t total_in = in_off[n];
    const uint8_t *d_in = nullptr;
    uint64_t *d_in_off = nullptr;
    if (stage_in(ctx->s_in, total_in + 16, in, total_in, st, &d_in) ||
        stage_in(ctx->s_in_off, (n + 1) * sizeof(uint64_t), in_off, n + 1, st, &d_in_off))
        return AWS_OP_ERR;
    aws_qpack_field_sections o{};
    o.n = n;
    o.field_capacity = field_capacity;
    o.strings_capacity = strings_capacity;
    if (stage_in(B.s_field_offsets, (n + 1) * sizeof(uint64_t), (const uint64_t *)nullptr, 0, st, &o.field_offsets) ||
        stage_in(B.s_eic, n * sizeof(uint64_t), (const uint64_t *)nullptr, 0, st, &o.encoded_insert_count) ||
        stage_in(B.s_sign, n, (const uint8_t *)nullptr, 0, st, &o.base_sign) ||
        stage_in(B.s_delta, n * sizeof(uint64_t), (const uint64_t *)nullptr, 0, st, &o.delta_base))
        return AWS_OP_ERR;
    HB_CUDA_TRY(ctx->s_status.reserve(n * sizeof(int32_t)));
    if (qpack_sections_decode_on_device(ctx, n, d_in, d_in_off, o, ctx->s_status.as<int32_t>(), true, st) ||
        read_back(o.field_offsets + n, &size[0], st))
        return AWS_OP_ERR;
    size[1] = 0;  // (string offsets exist for the fields that fit)
    return size[0] <= field_capacity ? read_back(B.s_string_offsets.as<uint64_t>() + 2 * size[0], &size[1], st) : AWS_OP_SUCCESS;
}

// Host pointers, finish into place: prefixes, offsets and status first (complete on AWS_ERROR_SHORT_BUFFER), then the
// records and strings.
int qpack_sections_decode_finish(
    aws_huffman_batch_ctx *ctx, size_t n, const uint64_t size[2], aws_qpack_field_sections *out, int32_t *status,
    cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    const uint64_t fields = size[0];
    HB_CUDA_TRY(cudaMemcpyAsync(out->encoded_insert_count, B.s_eic.ptr, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaMemcpyAsync(out->base_sign, B.s_sign.ptr, n, cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaMemcpyAsync(out->delta_base, B.s_delta.ptr, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (finish_slice(ctx, st, n, true, B.s_field_offsets.as<uint64_t>(), out->field_offsets, 0, nullptr, nullptr, 0, fields,
                     out->field_capacity, ctx->s_status.as<int32_t>(), status) ||
        finish_slice(ctx, st, 2 * fields, true, B.s_string_offsets.as<uint64_t>(), out->string_offsets, 0, ctx->s_out.ptr,
                     out->strings, size[1], size[1], out->strings_capacity))
        return AWS_OP_ERR;
    if (fields) {
        HB_CUDA_TRY(cudaMemcpyAsync(out->field_kind, B.s_kind.ptr, fields, cudaMemcpyDeviceToHost, st));
        HB_CUDA_TRY(cudaMemcpyAsync(out->field_index, B.s_index.ptr, fields * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        HB_CUDA_TRY(cudaMemcpyAsync(out->never_indexed, B.s_never.ptr, fields, cudaMemcpyDeviceToHost, st));
    }
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    return AWS_OP_SUCCESS;
}

// Arguments of the host-pointer decode call; a call with no sections is answered here (*done).
int qpack_sections_decode_args(size_t n, const uint8_t *in, const uint64_t *in_off, aws_qpack_field_sections *out, bool *done) {
    *done = false;
    if ((n && !in_off) || check_section_lists(out, true, false) || out->n != n) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (n == 0) {
        out->field_offsets[0] = 0;
        out->string_offsets[0] = 0;
        *done = true;
        return AWS_OP_SUCCESS;
    }
    if ((in_off[n] && !in) || !offsets_sorted(in_off, n + 1)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

int qpack_sections_decode_host(
    aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_off, aws_qpack_field_sections *out,
    int32_t *status) {
    bool done;
    if (!ctx) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (qpack_sections_decode_args(n, in, in_off, out, &done) || done) return done ? AWS_OP_SUCCESS : AWS_OP_ERR;
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    uint64_t size[2];
    int rc = qpack_sections_decode_slice(ctx, n, in, in_off, out->field_capacity, out->strings_capacity, size, st);
    if (rc == AWS_OP_SUCCESS) rc = qpack_sections_decode_finish(ctx, n, size, out, status, st);
    return call_end(ctx, st, rc);
}

// Host pointers, run on the device: the sections of `in` are staged and encoded into the context's staging,
// out_capacity octets at most; *size receives the output size. records: the kinds, indices and prefixes are read
// (aws_qpack_field_section_encode_records_batch) and a status per section is written to the staging.
int qpack_sections_encode_slice(
    aws_huffman_batch_ctx *ctx, const aws_qpack_field_sections *in, bool records, uint32_t mode, uint64_t out_capacity,
    uint64_t *size, cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    const uint64_t n = in->n, F = in->field_offsets[n], S = in->string_offsets[2 * F];
    uint64_t *d_field_offsets = nullptr, *d_string_offsets = nullptr;
    const uint8_t *d_strings = nullptr, *never = nullptr, *kind = nullptr, *sign = nullptr;
    const uint64_t *index = nullptr, *eic = nullptr, *delta = nullptr;
    int32_t *d_status = nullptr;
    if (records) {
        HB_CUDA_TRY(ctx->s_status.reserve(n * sizeof(int32_t)));
        d_status = ctx->s_status.as<int32_t>();
    }
    if (stage_in(B.s_field_offsets, (n + 1) * sizeof(uint64_t), in->field_offsets, n + 1, st, &d_field_offsets) ||
        stage_in(ctx->s_in, S + 16, in->strings, S, st, &d_strings) ||
        stage_in(ctx->s_in_off, (2 * F + 1) * sizeof(uint64_t), in->string_offsets, 2 * F + 1, st, &d_string_offsets) ||
        (in->never_indexed && F && stage_in(B.s_never, F, in->never_indexed, F, st, &never)) ||
        (records && (stage_in(B.s_kind, F + 1, in->field_kind, F, st, &kind) ||
                     stage_in(B.s_index, (F + 1) * sizeof(uint64_t), in->field_index, F, st, &index) ||
                     stage_in(B.s_eic, n * sizeof(uint64_t), in->encoded_insert_count, n, st, &eic) ||
                     stage_in(B.s_sign, n, in->base_sign, n, st, &sign) ||
                     stage_in(B.s_delta, n * sizeof(uint64_t), in->delta_base, n, st, &delta))))
        return AWS_OP_ERR;
    HB_CUDA_TRY(ctx->s_out.reserve(out_capacity + 16));
    HB_CUDA_TRY(ctx->s_out_off.reserve((n + 1) * sizeof(uint64_t)));
    if (qpack_sections_encode_on_device(ctx, n, d_field_offsets, F, never, kind, index, eic, sign, delta, d_strings,
                                        d_string_offsets, S, mode, ctx->s_out.as<uint8_t>(), out_capacity,
                                        ctx->s_out_off.as<uint64_t>(), d_status, st))
        return AWS_OP_ERR;
    return read_back(ctx->s_out_off.as<uint64_t>() + n, size, st);
}

// Arguments of the host-pointer encode calls (those of hpack_blocks_encode_args); a call with no sections is answered
// here (*done).
int qpack_sections_encode_args(const aws_qpack_field_sections *in, bool records, const uint8_t *out, uint64_t out_capacity,
                               uint64_t *out_off, bool *done) {
    *done = false;
    if (check_section_lists(in, false, records) || !out_off || (out_capacity && !out))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    const uint64_t n = in->n;
    if (n == 0) {
        out_off[0] = 0;
        *done = true;
        return AWS_OP_SUCCESS;
    }
    if (in->field_offsets[0] != 0 || !offsets_sorted(in->field_offsets, n + 1)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    const uint64_t F = in->field_offsets[n];
    if (in->string_offsets[0] != 0 || !offsets_sorted(in->string_offsets, 2 * F + 1))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (in->string_offsets[2 * F] && !in->strings) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

int qpack_sections_encode_host(
    aws_huffman_batch_ctx *ctx, const aws_qpack_field_sections *in, bool records, uint32_t mode, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_off, int32_t *status) {
    bool done;
    if (!ctx || mode > hb::kHpackAlways) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (qpack_sections_encode_args(in, records, out, out_capacity, out_off, &done) || done)
        return done ? AWS_OP_SUCCESS : AWS_OP_ERR;
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    uint64_t size = 0;
    int rc = qpack_sections_encode_slice(ctx, in, records, mode, out_capacity, &size, st);
    if (rc == AWS_OP_SUCCESS &&
        (finish_slice(ctx, st, in->n, true, ctx->s_out_off.as<uint64_t>(), out_off, 0, ctx->s_out.ptr, out, size, size,
                      out_capacity, records ? ctx->s_status.as<int32_t>() : nullptr, status) ||
         cudaStreamSynchronize(st) != cudaSuccess))
        rc = AWS_OP_ERR;
    return call_end(ctx, st, rc);
}

// ---------------------------------------------------------------------------------------------
// QPACK encoder- and decoder-stream instructions (qpack_instructions.cuh) over the passes and buffers of the field
// sections above. Device pointers in, device pointers out.
// ---------------------------------------------------------------------------------------------
// stage: `o` holds instruction_offsets (context staging) and the capacities; the per-instruction outputs go to context
// staging sized from the totals (the host entry point copies them back).
int qpack_instructions_decode_on_device(
    aws_huffman_batch_ctx *ctx, uint32_t which, uint64_t n, const uint8_t *in, const uint64_t *in_off,
    aws_qpack_instructions o, uint64_t *consumed, int32_t *status, bool stage, cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    if (n == 0) {
        HB_CUDA_TRY(cudaMemsetAsync(o.instruction_offsets, 0, sizeof(uint64_t), st));
        if (o.string_offsets && !stage) HB_CUDA_TRY(cudaMemsetAsync(o.string_offsets, 0, sizeof(uint64_t), st));
        return AWS_OP_SUCCESS;
    }
    const unsigned flat = grid_of(n, 256);
    HB_CUDA_TRY(B.num_fields.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.num_lits.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_bytes.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.out_fields.reserve(n * sizeof(uint64_t)));
    HB_CUDA_TRY(B.struct_status.reserve(n * sizeof(int32_t)));
    HB_CUDA_TRY(B.field_base.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_base.reserve((n + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_byte_base.reserve((n + 1) * sizeof(uint64_t)));
    if (!status) {
        HB_CUDA_TRY(B.status.reserve(n * sizeof(int32_t)));
        status = B.status.as<int32_t>();
    }
    if (!B.h_totals) HB_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&B.h_totals), 3 * sizeof(uint64_t), cudaHostAllocDefault));
    uint64_t *instr_base = B.field_base.as<uint64_t>(), *lit_base = B.lit_base.as<uint64_t>();
    uint64_t *lit_byte_base = B.lit_byte_base.as<uint64_t>();

    // 1. structure, counts, consumed lengths; 2. their bases, and the totals the later launches are sized from
    hb::qpack_instruction_scan_kernel<<<flat, 256, 0, st>>>(n, which, in, in_off, B.num_fields.as<uint64_t>(),
                                                             B.num_lits.as<uint64_t>(), B.lit_bytes.as<uint64_t>(), consumed,
                                                             B.struct_status.as<int32_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.num_fields.as<uint64_t>(), instr_base, n, st)) return AWS_OP_ERR;
    if (launch_scan(ctx, ctx->scratch, B.num_lits.as<uint64_t>(), lit_base, n, st)) return AWS_OP_ERR;
    if (launch_scan(ctx, ctx->scratch, B.lit_bytes.as<uint64_t>(), lit_byte_base, n, st)) return AWS_OP_ERR;
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 0, instr_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 1, lit_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaMemcpyAsync(B.h_totals + 2, lit_byte_base + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    const uint64_t parsed = B.h_totals[0], num_lits = B.h_totals[1], lit_total = B.h_totals[2];
    const uint64_t kept = std::min(parsed, o.instruction_capacity);  // instruction slots that can be written
    const uint32_t min_len = std::max<uint32_t>(1, ctx->tables.min_len);
    const uint64_t dec_cap = lit_total * 8 / min_len + 64;
    if (stage) {
        // (an instruction's strings are its decoded literals or an Appendix A name, at most 32 octets)
        o.strings_capacity = std::min(o.strings_capacity, dec_cap + 32 * kept);
        HB_CUDA_TRY(B.s_kind.reserve(kept + 1));
        HB_CUDA_TRY(B.s_index.reserve((kept + 1) * sizeof(uint64_t)));
        HB_CUDA_TRY(B.s_string_offsets.reserve((2 * kept + 1) * sizeof(uint64_t)));
        HB_CUDA_TRY(ctx->s_out.reserve(o.strings_capacity + 16));
        o.kind = B.s_kind.as<uint8_t>();
        o.index = B.s_index.as<uint64_t>();
        o.string_offsets = B.s_string_offsets.as<uint64_t>();
        o.strings = ctx->s_out.as<uint8_t>();
    }
    HB_CUDA_TRY(B.f_kind.reserve(parsed + 1));
    HB_CUDA_TRY(B.f_index.reserve((parsed + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.f_block.reserve((parsed + 1) * sizeof(uint32_t)));
    HB_CUDA_TRY(B.f_lits.reserve((2 * parsed + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_src.reserve((num_lits + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_len.reserve((num_lits + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_offsets.reserve((num_lits + 1) * sizeof(uint64_t)));
    HB_CUDA_TRY(B.lit_status.reserve((num_lits + 1) * sizeof(int32_t)));
    HB_CUDA_TRY(B.dec_offsets.reserve((num_lits + 1) * sizeof(uint64_t)));
    uint8_t *f_kind = B.f_kind.as<uint8_t>();
    uint64_t *f_index = B.f_index.as<uint64_t>(), *f_lits = B.f_lits.as<uint64_t>();
    uint32_t *f_block = B.f_block.as<uint32_t>();
    uint64_t *dec_offsets = B.dec_offsets.as<uint64_t>();
    int32_t *lit_status = B.lit_status.as<int32_t>();

    // 3. instruction records and literals in parsed order; 4. the literals, packed and re-framed as RFC 7541 5.2
    // literals; 5. decoded by the literal path (a decoder-stream batch has no literals)
    if (parsed || num_lits) {
        hb::qpack_instruction_split_kernel<<<flat, 256, 0, st>>>(
            n, which, in, in_off, instr_base, lit_base, lit_byte_base, f_kind, f_index, f_block, f_lits,
            B.lit_src.as<uint64_t>(), B.lit_len.as<uint64_t>(), B.lit_offsets.as<uint64_t>());
        ++ctx->launches;
    }
    if (num_lits) {
        HB_CUDA_TRY(B.lits.reserve(lit_total + 64));
        HB_CUDA_TRY(B.dec.reserve(dec_cap + 64));
        hb::qpack_lit_gather_kernel<<<grid_of(num_lits, 256), 256, 0, st>>>(
            num_lits, in, B.lit_src.as<uint64_t>(), B.lit_len.as<uint64_t>(), B.lit_offsets.as<uint64_t>(), B.lits.as<uint8_t>());
        ++ctx->launches;
        if (hpack_decode_on_device(ctx, num_lits, B.lits.as<uint8_t>(), B.lit_offsets.as<uint64_t>(), lit_total,
                                   B.dec.as<uint8_t>(), dec_cap, dec_offsets, lit_status, st))
            return AWS_OP_ERR;
    }
    // 6. final status per chunk, consumed lengths, instruction offsets; 7. records, string lengths, string offsets,
    // strings
    hb::hpack_block_finish_kernel<<<flat, 256, 0, st>>>(
        n, lit_base, lit_status, B.struct_status.as<int32_t>(), B.num_fields.as<uint64_t>(), status, B.out_fields.as<uint64_t>());
    ++ctx->launches;
    hb::qpack_instruction_consumed_kernel<<<flat, 256, 0, st>>>(n, status, consumed);
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.out_fields.as<uint64_t>(), o.instruction_offsets, n, st)) return AWS_OP_ERR;
    if (!kept) {
        HB_CUDA_TRY(cudaMemsetAsync(o.string_offsets, 0, sizeof(uint64_t), st));
        HB_CUDA_TRY(cudaGetLastError());
        return AWS_OP_SUCCESS;
    }
    HB_CUDA_TRY(B.str_lens.reserve(2 * kept * sizeof(uint64_t)));
    HB_CUDA_TRY(cudaMemsetAsync(B.str_lens.ptr, 0, 2 * kept * sizeof(uint64_t), st));
    const uint8_t *dec = B.dec.as<uint8_t>();
    hb::hpack_field_records_kernel<hb::QpackInstructionStrings><<<grid_of(parsed, 256), 256, 0, st>>>(
        parsed, f_kind, f_index, f_block, f_lits, instr_base, status, o.instruction_offsets, o.instruction_capacity, dec,
        dec_offsets, o.kind, o.index, B.str_lens.as<uint64_t>());
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.str_lens.as<uint64_t>(), o.string_offsets, 2 * kept, st)) return AWS_OP_ERR;
    hb::hpack_compose_kernel<hb::QpackInstructionStrings><<<grid_of(2 * parsed, 256), 256, 0, st>>>(
        parsed, f_kind, f_index, f_block, f_lits, instr_base, status, o.instruction_offsets, o.instruction_capacity, dec,
        dec_offsets, o.strings, o.strings_capacity, o.string_offsets);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// The caller's instructions (kind, index; names and values on the encoder stream) into n chunks of the stream `which`,
// with the per-chunk status (optional) of aws_qpack_instruction_encode_batch.
int qpack_instructions_encode_on_device(
    aws_huffman_batch_ctx *ctx, uint32_t which, uint64_t n, const uint64_t *instruction_offsets, uint64_t num_instr,
    const uint8_t *kind, const uint64_t *index, const uint8_t *strings, const uint64_t *string_offsets,
    uint64_t strings_size, uint32_t mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status,
    cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    if (n == 0 || num_instr == 0) {
        HB_CUDA_TRY(cudaMemsetAsync(out_offsets, 0, (n + 1) * sizeof(uint64_t), st));
        if (status && n) HB_CUDA_TRY(cudaMemsetAsync(status, 0, n * sizeof(int32_t), st));
        return AWS_OP_SUCCESS;
    }
    const uint64_t F = num_instr;
    HB_CUDA_TRY(B.plan.reserve(F));
    HB_CUDA_TRY(B.plan_index.reserve(F * sizeof(uint64_t)));
    HB_CUDA_TRY(B.field_lens.reserve(F * sizeof(uint64_t)));
    HB_CUDA_TRY(B.field_pos.reserve((F + 1) * sizeof(uint64_t)));
    uint64_t *field_pos = B.field_pos.as<uint64_t>();
    const uint8_t *framed = nullptr;
    const uint64_t *framed_offsets = nullptr;
    // 1. every name and value framed (encoder stream: the decoder stream sends no literals); 2. instruction and size;
    // 3. the chunk rule; 4. wire positions of instructions and chunks; 5. the instructions
    if (which == 0) {
        const uint64_t expand = mode == hb::kHpackAlways ? (std::max<uint32_t>(1, ctx->tables.max_len) + 7) / 8 : 1;
        const uint64_t framed_cap = strings_size * expand + 2 * F * 10 + 64;
        HB_CUDA_TRY(B.framed.reserve(framed_cap + 64));
        HB_CUDA_TRY(B.framed_offsets.reserve((2 * F + 1) * sizeof(uint64_t)));
        framed = B.framed.as<uint8_t>();
        framed_offsets = B.framed_offsets.as<uint64_t>();
        if (hpack_encode_on_device(ctx, 2 * F, strings, string_offsets, strings_size, mode, B.framed.as<uint8_t>(),
                                   framed_cap, B.framed_offsets.as<uint64_t>(), st))
            return AWS_OP_ERR;
    }
    hb::qpack_instruction_plan_kernel<<<grid_of(F, 256), 256, 0, st>>>(
        F, which, strings, string_offsets, kind, index, framed, framed_offsets, B.plan.as<uint8_t>(),
        B.plan_index.as<uint64_t>(), B.field_lens.as<uint64_t>());
    ++ctx->launches;
    hb::qpack_instruction_check_kernel<<<grid_of(n, 256), 256, 0, st>>>(n, instruction_offsets, B.plan.as<uint8_t>(),
                                                                         B.field_lens.as<uint64_t>(), status);
    ++ctx->launches;
    if (launch_scan(ctx, ctx->scratch, B.field_lens.as<uint64_t>(), field_pos, F, st)) return AWS_OP_ERR;
    hb::hpack_block_offsets_kernel<<<grid_of(n + 1, 256), 256, 0, st>>>(n, instruction_offsets, field_pos, out_offsets);
    ++ctx->launches;
    hb::qpack_field_emit_kernel<hb::QpackInstructionLines><<<grid_of(F, 256), 256, 0, st>>>(
        F, B.plan.as<uint8_t>(), B.plan_index.as<uint64_t>(), framed, framed_offsets, field_pos, out, out_capacity);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

// The argument rules of the instruction calls that need no device memory read. Decode writes kind, index, strings and
// string_offsets; encode reads kind and index, and on the encoder stream string_offsets.
int check_instruction_lists(const aws_qpack_instructions *l, uint32_t which, bool decode) {
    if (!l || which > 1 || (l->n && !l->instruction_offsets) || l->n > 0xffffffffull)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (decode && (!l->string_offsets || (l->instruction_capacity && (!l->kind || !l->index)) ||
                   (l->strings_capacity && !l->strings)))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (!decode && (!l->kind || !l->index || (which == 0 && !l->string_offsets)))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

// Host pointers, run on the device (the way qpack_sections_decode_slice does): the n chunks are staged and decoded
// into the context's staging, within the capacities given; size[0] receives their instructions and, when those fit
// instruction_capacity, size[1] their string octets.
int qpack_instructions_decode_slice(
    aws_huffman_batch_ctx *ctx, uint32_t which, size_t n, const uint8_t *in, const uint64_t *in_off,
    uint64_t instruction_capacity, uint64_t strings_capacity, uint64_t size[2], cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    const uint64_t total_in = in_off[n];
    const uint8_t *d_in = nullptr;
    uint64_t *d_in_off = nullptr, *d_consumed = nullptr;
    aws_qpack_instructions o{};
    o.n = n;
    o.instruction_capacity = instruction_capacity;
    o.strings_capacity = strings_capacity;
    if (stage_in(ctx->s_in, total_in + 16, in, total_in, st, &d_in) ||
        stage_in(ctx->s_in_off, (n + 1) * sizeof(uint64_t), in_off, n + 1, st, &d_in_off) ||
        stage_in(B.s_field_offsets, (n + 1) * sizeof(uint64_t), (const uint64_t *)nullptr, 0, st, &o.instruction_offsets) ||
        stage_in(ctx->s_consumed, n * sizeof(uint64_t), (const uint64_t *)nullptr, 0, st, &d_consumed))
        return AWS_OP_ERR;
    HB_CUDA_TRY(ctx->s_status.reserve(n * sizeof(int32_t)));
    if (qpack_instructions_decode_on_device(ctx, which, n, d_in, d_in_off, o, d_consumed, ctx->s_status.as<int32_t>(),
                                            true, st) ||
        read_back(o.instruction_offsets + n, &size[0], st))
        return AWS_OP_ERR;
    size[1] = 0;  // (string offsets exist for the instructions that fit)
    return size[0] <= instruction_capacity ? read_back(B.s_string_offsets.as<uint64_t>() + 2 * size[0], &size[1], st)
                                           : AWS_OP_SUCCESS;
}

// Host pointers, finish into place: consumed lengths, offsets and status first (complete on AWS_ERROR_SHORT_BUFFER),
// then the records and strings.
int qpack_instructions_decode_finish(
    aws_huffman_batch_ctx *ctx, size_t n, const uint64_t size[2], aws_qpack_instructions *out, uint64_t *consumed,
    int32_t *status, cudaStream_t st) {
    hb_host::BlockBufs &B = ctx->blk;
    const uint64_t instr = size[0];
    HB_CUDA_TRY(cudaMemcpyAsync(consumed, ctx->s_consumed.ptr, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (finish_slice(ctx, st, n, true, B.s_field_offsets.as<uint64_t>(), out->instruction_offsets, 0, nullptr, nullptr, 0,
                     instr, out->instruction_capacity, ctx->s_status.as<int32_t>(), status) ||
        finish_slice(ctx, st, 2 * instr, true, B.s_string_offsets.as<uint64_t>(), out->string_offsets, 0, ctx->s_out.ptr,
                     out->strings, size[1], size[1], out->strings_capacity))
        return AWS_OP_ERR;
    if (instr) {
        HB_CUDA_TRY(cudaMemcpyAsync(out->kind, B.s_kind.ptr, instr, cudaMemcpyDeviceToHost, st));
        HB_CUDA_TRY(cudaMemcpyAsync(out->index, B.s_index.ptr, instr * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    }
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    return AWS_OP_SUCCESS;
}

int qpack_instructions_decode_host(
    aws_huffman_batch_ctx *ctx, uint32_t which, size_t n, const uint8_t *in, const uint64_t *in_off,
    aws_qpack_instructions *out, uint64_t *consumed, int32_t *status) {
    if (!ctx || (n && (!in_off || !consumed)) || check_instruction_lists(out, which, true) || out->n != n)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (n == 0) {
        out->instruction_offsets[0] = 0;
        out->string_offsets[0] = 0;
        return AWS_OP_SUCCESS;
    }
    if ((in_off[n] && !in) || !offsets_sorted(in_off, n + 1)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    uint64_t size[2];
    int rc = qpack_instructions_decode_slice(ctx, which, n, in, in_off, out->instruction_capacity, out->strings_capacity,
                                             size, st);
    if (rc == AWS_OP_SUCCESS) rc = qpack_instructions_decode_finish(ctx, n, size, out, consumed, status, st);
    return call_end(ctx, st, rc);
}

// Host pointers: the chunks of `in` are staged and encoded into the context's staging, out_capacity octets at most;
// *size receives the output size and the status per chunk goes to the staging.
int qpack_instructions_encode_slice(
    aws_huffman_batch_ctx *ctx, uint32_t which, const aws_qpack_instructions *in, uint32_t mode, uint64_t out_capacity,
    uint64_t *size, cudaStream_t st) {
    const uint64_t n = in->n, F = in->instruction_offsets[n], S = which == 0 ? in->string_offsets[2 * F] : 0;
    hb_host::BlockBufs &B = ctx->blk;
    uint64_t *d_offsets = nullptr, *d_string_offsets = nullptr;
    const uint8_t *d_strings = nullptr, *d_kind = nullptr;
    const uint64_t *d_index = nullptr;
    HB_CUDA_TRY(ctx->s_status.reserve(n * sizeof(int32_t)));
    if (stage_in(B.s_field_offsets, (n + 1) * sizeof(uint64_t), in->instruction_offsets, n + 1, st, &d_offsets) ||
        stage_in(B.s_kind, F + 1, in->kind, F, st, &d_kind) ||
        stage_in(B.s_index, (F + 1) * sizeof(uint64_t), in->index, F, st, &d_index) ||
        (which == 0 && (stage_in(ctx->s_in, S + 16, in->strings, S, st, &d_strings) ||
                        stage_in(ctx->s_in_off, (2 * F + 1) * sizeof(uint64_t), in->string_offsets, 2 * F + 1, st,
                                 &d_string_offsets))))
        return AWS_OP_ERR;
    HB_CUDA_TRY(ctx->s_out.reserve(out_capacity + 16));
    HB_CUDA_TRY(ctx->s_out_off.reserve((n + 1) * sizeof(uint64_t)));
    if (qpack_instructions_encode_on_device(ctx, which, n, d_offsets, F, d_kind, d_index, d_strings, d_string_offsets, S,
                                            mode, ctx->s_out.as<uint8_t>(), out_capacity, ctx->s_out_off.as<uint64_t>(),
                                            ctx->s_status.as<int32_t>(), st))
        return AWS_OP_ERR;
    return read_back(ctx->s_out_off.as<uint64_t>() + n, size, st);
}

int qpack_instructions_encode_host(
    aws_huffman_batch_ctx *ctx, uint32_t which, const aws_qpack_instructions *in, uint32_t mode, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_off, int32_t *status) {
    if (!ctx || mode > hb::kHpackAlways || check_instruction_lists(in, which, false) || !out_off ||
        (out_capacity && !out))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    const uint64_t n = in->n;
    if (n == 0) {
        out_off[0] = 0;
        return AWS_OP_SUCCESS;
    }
    // (instructions are numbered from 0 and every one is encoded: chunks start at instruction 0, strings at octet 0)
    if (in->instruction_offsets[0] != 0 || !offsets_sorted(in->instruction_offsets, n + 1))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    const uint64_t F = in->instruction_offsets[n];
    if (which == 0 && (in->string_offsets[0] != 0 || !offsets_sorted(in->string_offsets, 2 * F + 1) ||
                       (in->string_offsets[2 * F] && !in->strings)))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    uint64_t size = 0;
    int rc = qpack_instructions_encode_slice(ctx, which, in, mode, out_capacity, &size, st);
    if (rc == AWS_OP_SUCCESS &&
        (finish_slice(ctx, st, n, true, ctx->s_out_off.as<uint64_t>(), out_off, 0, ctx->s_out.ptr, out, size, size,
                      out_capacity, ctx->s_status.as<int32_t>(), status) ||
         cudaStreamSynchronize(st) != cudaSuccess))
        rc = AWS_OP_ERR;
    return call_end(ctx, st, rc);
}

// ---------------------------------------------------------------------------------------------
// Byte histogram (SURVEY.md 8f.4: the counts a code table is built from). HBM-bound by construction: 16 bytes per
// lane and load, and a block-wide histogram with ONE COLUMN PER LANE (hist[value][lane]): the 32 lanes of a
// shared-memory atomic never meet in an address and every lane stays in its own bank, however skewed the
// data is (the benchmark's top symbol is 40 % of the bytes: per-warp histograms would serialise 13-fold).
// ---------------------------------------------------------------------------------------------
constexpr int kHistThreads = 512;

__global__ void __launch_bounds__(kHistThreads) histogram_kernel(const uint8_t *in, uint64_t size, unsigned long long *counts) {
    __shared__ uint32_t s_hist[256 * 32];
    for (uint32_t i = threadIdx.x; i < 256 * 32; i += kHistThreads) s_hist[i] = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    uint32_t *const mine = s_hist + lane;
    const uintptr_t base = reinterpret_cast<uintptr_t>(in);
    const uint64_t head = min((unsigned long long)size, (unsigned long long)((16 - (base & 15)) & 15));  // bytes before the first aligned 16
    const uint64_t nvec = (size - head) >> 4;
    const uint4 *v = reinterpret_cast<const uint4 *>(in + head);
    auto add_word = [&](uint32_t w) {
        atomicAdd(mine + ((w & 0xffu) << 5), 1u);
        atomicAdd(mine + (((w >> 8) & 0xffu) << 5), 1u);
        atomicAdd(mine + (((w >> 16) & 0xffu) << 5), 1u);
        atomicAdd(mine + ((w >> 24) << 5), 1u);
    };
    for (uint64_t i = (uint64_t)blockIdx.x * kHistThreads + threadIdx.x; i < nvec; i += (uint64_t)gridDim.x * kHistThreads) {
        const uint4 q = __ldg(v + i);
        add_word(q.x);
        add_word(q.y);
        add_word(q.z);
        add_word(q.w);
    }
    if (blockIdx.x == 0) {  // the ragged ends
        const uint64_t tail0 = head + 16 * nvec;
        for (uint64_t i = threadIdx.x; i < head; i += kHistThreads) atomicAdd(mine + ((uint32_t)in[i] << 5), 1u);
        for (uint64_t i = tail0 + threadIdx.x; i < size; i += kHistThreads) atomicAdd(mine + ((uint32_t)in[i] << 5), 1u);
    }
    __syncthreads();
    // 256 values x 32 columns -> one count per value (a warp per value, 16 values per warp)
    for (uint32_t value = threadIdx.x >> 5; value < 256; value += kHistThreads / 32) {
        uint32_t c = s_hist[value * 32 + lane];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
        if (lane == 0 && c) atomicAdd(counts + value, (unsigned long long)c);
    }
}

int histogram_on_device(const uint8_t *in, uint64_t size, uint64_t *counts, cudaStream_t st) {
    HB_CUDA_TRY(cudaMemsetAsync(counts, 0, 256 * sizeof(uint64_t), st));
    if (size == 0) return AWS_OP_SUCCESS;
    int device = 0, sms = 148;
    HB_CUDA_TRY(cudaGetDevice(&device));
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    // (a block's 32-bit columns hold its share of the bytes: size / blocks / 32 per column at most)
    const uint64_t want = (size / 16 + kHistThreads - 1) / kHistThreads;
    const unsigned blocks = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(want, (uint64_t)sms * 4));
    histogram_kernel<<<blocks, kHistThreads, 0, st>>>(in, size, reinterpret_cast<unsigned long long *>(counts));
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

__global__ void encoded_length_kernel(hb::DeviceTables t, const uint8_t *in, const uint64_t *in_offsets, uint64_t n, uint64_t *lens) {
    __shared__ uint32_t s_len[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_len[i] = t.enc[i].y;
    __syncthreads();
    const uint64_t item = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= n) return;
    const uint64_t a = in_offsets[item], e = in_offsets[item + 1];
    uint64_t bits = 0;
    for (uint64_t k = a + hb::lane_id(); k < e; k += 32) bits += s_len[in[k]];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) bits += __shfl_xor_sync(0xffffffffu, bits, d);
    if (hb::lane_id() == 0) lens[item] = (bits + 7) >> 3;
}

int encoded_lengths_on_device(
    aws_huffman_batch_ctx *ctx, const uint8_t *in, const uint64_t *in_offsets, size_t n, uint64_t *lens, cudaStream_t st) {
    const unsigned blocks = (unsigned)((n + kWarpsPerBlock - 1) / kWarpsPerBlock);
    encoded_length_kernel<<<blocks, kWarpsPerBlock * 32, 0, st>>>(ctx->tables, in, in_offsets, n, lens);
    ++ctx->launches;
    HB_CUDA_TRY(cudaGetLastError());
    return AWS_OP_SUCCESS;
}

int encoded_lengths_staged(
    aws_huffman_batch_ctx *ctx, const uint8_t *in, const uint64_t *in_offsets, size_t n, uint64_t *lens, cudaStream_t st) {
    const uint64_t total_in = in_offsets[n];
    const uint8_t *d_in = nullptr;
    const uint64_t *d_in_off = nullptr;
    uint64_t *d_lens = nullptr;
    if (stage_in(ctx->s_in, total_in + 16, in, total_in, st, &d_in) ||
        stage_in(ctx->s_in_off, (n + 1) * sizeof(uint64_t), in_offsets, n + 1, st, &d_in_off) ||
        stage_in(ctx->scratch.lens, n * sizeof(uint64_t), lens, 0, st, &d_lens) ||
        encoded_lengths_on_device(ctx, d_in, d_in_off, n, d_lens, st))
        return AWS_OP_ERR;
    HB_CUDA_TRY(cudaMemcpyAsync(lens, d_lens, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA_TRY(cudaStreamSynchronize(st));
    return AWS_OP_SUCCESS;
}

// What the launches need that depends only on the device and the code table, worked out once per context. The
// dynamic shared-memory limits are the same for every context on a device (the encoders' compile-time sizes; the
// decoders get all the device allows beside what they declare), so no context can lower another one's.
int configure_kernels(aws_huffman_batch_ctx *ctx) {
    constexpr cudaFuncAttribute kLimit = cudaFuncAttributeMaxDynamicSharedMemorySize;
    int sms = 0, optin = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device) == cudaSuccess && sms > 0)
        ctx->sm_count = sms;
    HB_CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));

    HB_CUDA_TRY(cudaFuncSetAttribute(encode_tiled_kernel<false>, kLimit, (int)kEncSmemBytes));
    HB_CUDA_TRY(cudaFuncSetAttribute(encode_tiled_kernel<true>, kLimit, (int)kEncSmemBytes));
    HB_CUDA_TRY(cudaFuncSetAttribute(encode_slots_kernel, kLimit, (int)kEncSlotSmemBytes));
    HB_CUDA_TRY(cudaFuncSetAttribute(str_pack_kernel, kLimit, (int)kStrPackSmemBytes));
    HB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->enc_blocks_per_sm[0], encode_tiled_kernel<false>, kEncBlock, kEncSmemBytes));
    HB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->enc_blocks_per_sm[1], encode_tiled_kernel<true>, kEncBlock, kEncSmemBytes));
    HB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->enc_slots_blocks_per_sm, encode_slots_kernel, kEncBlock, kEncSlotSmemBytes));
    HB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->str_blocks_per_sm[0], str_bits_kernel, kBitsThreads, 0));
    HB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->str_blocks_per_sm[1], str_pack_kernel, kStrThreads, kStrPackSmemBytes));
    for (int *per_sm : {&ctx->enc_blocks_per_sm[0], &ctx->enc_blocks_per_sm[1], &ctx->enc_slots_blocks_per_sm,
                        &ctx->str_blocks_per_sm[0], &ctx->str_blocks_per_sm[1]})
        *per_sm = std::max(1, *per_sm);

    size_t declared[2] = {0, 0};  // static shared memory of decode_batch_kernel<framed>
    auto open_up = [&](auto kernel, size_t *static_smem) -> int {
        cudaFuncAttributes attr{};
        HB_CUDA_TRY(cudaFuncGetAttributes(&attr, kernel));
        if (static_smem) *static_smem = attr.sharedSizeBytes;
        HB_CUDA_TRY(cudaFuncSetAttribute(kernel, kLimit, optin - (int)attr.sharedSizeBytes));
        return AWS_OP_SUCCESS;
    };
    if (open_up(decode_batch_kernel<false>, &declared[0]) || open_up(decode_batch_kernel<true>, &declared[1]) ||
        open_up(stream_fused_kernel, nullptr) || open_up(stream_sync_kernel, nullptr) || open_up(stream_write_kernel, nullptr))
        return AWS_OP_ERR;

    // decode_batch_fast. Shared memory of one block (two blocks per SM): [LUT][stage][rows]. A string of L bytes
    // decodes to at most 8 L / min_len symbols, so the row area is that much larger than the stage; and the dense
    // output image (which reuses the stage and the front of the rows) must end before row offset `front`
    // (decode_batch_kernel step 4): rows <= stage + front - 32.
    const uint32_t min_len = std::max<uint32_t>(1, ctx->tables.min_len);
    const size_t lut_bytes = (size_t)ctx->lut2_count * 8;
    for (int framed = 0; framed < 2; ++framed) {
        // one block per SM: [LUT2][team 0: stage, rows][team 1: stage, rows] + the teams' static arrays (what the
        // kernel declares is asked from the runtime: every KB of the SM's 227 is a string more per tile)
        const size_t budget = (((size_t)227 * 1024 - declared[framed] - lut_bytes) / kDecTeams - 128) & ~size_t(15);
        const double expand = 8.0 / min_len;
        size_t stage_bytes = (size_t)((double)budget / (1.0 + expand)) & ~size_t(15);
        stage_bytes = std::max<size_t>(stage_bytes, 2 * kDecMaxRow);
        size_t rows_bytes = budget - stage_bytes;
        const size_t front = (stage_bytes - kDecMaxRow - 32) & ~size_t(3);
        rows_bytes = std::min(rows_bytes, stage_bytes + front - 64) & ~size_t(15);
        const size_t team_bytes = ((stage_bytes + 15) & ~size_t(15)) + rows_bytes + 64;
        ctx->dec_layout[framed] = {stage_bytes, rows_bytes, lut_bytes + kDecTeams * team_bytes};
    }

    // decode_stream_fast
    hb_host::StreamLayout &S = ctx->stream_layout;
    S.smem = ctx->tables.lut_count * sizeof(uint32_t);
    S.smem_staged = S.smem + kStreamStageWords * sizeof(uint32_t);
    S.row_words = (((kChunkBits + 31) / min_len + 4 + 3) / 4) | 1u;
    const size_t stage_bytes = (kStreamStageWords * 4 + 15) & ~size_t(15);
    const size_t team_bytes = (stage_bytes + (size_t)kStreamThreads * S.row_words * 4 + 16 + 15) & ~size_t(15);
    S.fused_smem = lut_bytes + kStreamTeams * team_bytes;  // one block per SM, two teams, one table
    // (the dense output image reuses the stage and the front of the rows: stream_fused_kernel step 5)
    S.fused = (size_t)kStreamThreads * S.row_words * 4 + 16 <= 2 * stage_bytes - S.row_words * 4 - 32 &&
              S.fused_smem <= 220 * 1024 && !ctx->no_fused_stream;
    return AWS_OP_SUCCESS;
}

// ---------------------------------------------------------------------------------------------
// One host-pointer call over several contexts (the _multi entry points): the items are cut into one contiguous range
// per context, balanced by bytes (aws_huffman_batch_plan_shards), and each range runs on a host thread of its own.
// No collective: the shards never talk to each other.
// ---------------------------------------------------------------------------------------------
int check_contexts(aws_huffman_batch_ctx *const *ctxs, size_t n_ctx) {
    if (!ctxs || n_ctx == 0) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    for (size_t d = 0; d < n_ctx; ++d)
        if (!ctxs[d]) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return AWS_OP_SUCCESS;
}

// shard(d) for d in [0, n_ctx), each on a thread of its own. The error slot is per thread, so every shard's error is
// collected there; the first shard in item order that failed decides the call's error, whichever finished first.
template <typename Shard>
int run_shards(size_t n_ctx, const Shard &shard) {
    std::vector<int> err(n_ctx, 0);
    std::vector<std::thread> threads;
    for (size_t d = 0; d < n_ctx; ++d) {
        threads.emplace_back([&, d]() {
            if (shard(d) != AWS_OP_SUCCESS) err[d] = aws_last_error() ? aws_last_error() : AWS_ERROR_COMPRESSION_DEVICE_FAILURE;
        });
    }
    for (std::thread &t : threads) t.join();
    for (int e : err)
        if (e) return aws_raise_error(e);
    return AWS_OP_SUCCESS;
}

// Output totals of one shard: octets out, or fields and string octets.
using Totals = std::array<uint64_t, 2>;

// Where the shard threads of one call meet after running their shards on the device: every thread publishes its
// totals, or its failure, exactly once and waits for all the others (an empty shard publishes at once, a failed one
// too, so no thread waits forever). Each leaves with the same totals, so each finds its own bases and reaches the
// capacity decision the single-context call reaches.
class ShardExchange {
  public:
    explicit ShardExchange(size_t shards) : totals_(shards), waiting_(shards) {}
    // false when some shard failed: then no shard writes the caller's arrays
    bool publish(size_t shard, bool ok, const Totals &totals) {
        std::unique_lock<std::mutex> lock(mutex_);
        totals_[shard] = totals;
        failed_ |= !ok;
        if (--waiting_ == 0) all_in_.notify_all();
        else all_in_.wait(lock, [this] { return waiting_ == 0; });
        return !failed_;
    }
    // (after publish) the sum over the shards before `shard`, i.e. its bases, and over all of them
    Totals before(size_t shard) const {
        Totals sum{0, 0};
        for (size_t s = 0; s < shard; ++s)
            for (size_t k = 0; k < sum.size(); ++k) sum[k] += totals_[s][k];
        return sum;
    }
    Totals all() const { return before(totals_.size()); }

  private:
    std::vector<Totals> totals_;
    size_t waiting_;
    bool failed_ = false;
    std::mutex mutex_;
    std::condition_variable all_in_;
};

// An HPACK host-pointer call over several contexts, its shards planned on `weight` (n + 1 non-decreasing values).
// Each shard's thread runs its slice on the device straight from the caller's arrays (run: shard totals out), meets
// the others, and copies its offsets, status, records and payload into the caller's arrays at its bases (finish): no
// host-side copy or concatenation of the per-item arrays.
//     run(ctx, first, count, uint64_t *size, st)
//     finish(ctx, first, count, bool last, const uint64_t *base, const uint64_t *size, const uint64_t *total, st)
template <typename Run, typename Finish>
int hpack_multi(aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, size_t n, const uint64_t *weight, const Run &run,
                const Finish &finish) {
    std::vector<size_t> begin(n_ctx + 1);
    if (aws_huffman_batch_plan_shards(weight, n, n_ctx, begin.data())) return AWS_OP_ERR;
    ShardExchange exchange(n_ctx);
    return run_shards(n_ctx, [&](size_t d) -> int {
        aws_huffman_batch_ctx *ctx = ctxs[d];
        const size_t first = begin[d], count = begin[d + 1] - first;
        Totals size{0, 0};
        if (count == 0) {  // no device work
            exchange.publish(d, true, size);
            return AWS_OP_SUCCESS;
        }
        cudaStream_t st;
        if (call_begin(ctx, nullptr, &st)) {
            exchange.publish(d, false, size);
            return AWS_OP_ERR;
        }
        int rc = run(ctx, first, count, size.data(), st);
        if (exchange.publish(d, rc == AWS_OP_SUCCESS, size)) {
            const Totals base = exchange.before(d), total = exchange.all();
            rc = finish(ctx, first, count, first + count == n, base.data(), size.data(), total.data(), st);
        }
        return call_end(ctx, st, rc);
    });
}

int hpack_literals_multi(
    aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, bool encode, size_t n, const uint8_t *in, const uint64_t *in_off,
    uint32_t mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_off, int32_t *status) {
    bool done;
    if (check_contexts(ctxs, n_ctx)) return AWS_OP_ERR;
    if (n_ctx == 1) return hpack_run_host(ctxs[0], encode, n, in, in_off, mode, out, out_capacity, out_off, status);
    if (hpack_host_args(n, in, in_off, out, out_capacity, out_off, &done) || done) return done ? AWS_OP_SUCCESS : AWS_OP_ERR;
    auto run = [&](aws_huffman_batch_ctx *ctx, size_t first, size_t count, uint64_t *size, cudaStream_t st) {
        // the shard's staging holds all its output: framed, a prefix of at most 10 octets and a payload no longer than
        // the string unless every literal is Huffman-coded; decoded, a raw payload or at most 8 / min_len symbols an octet
        const uint64_t bytes = in_off[first + count] - in_off[first];
        const uint64_t expand = mode == hb::kHpackAlways ? (std::max<uint32_t>(1, ctx->tables.max_len) + 7) / 8 : 1;
        const uint64_t room = encode ? bytes * expand + 10 * (uint64_t)count + 64
                                     : bytes * 8 / std::min<uint32_t>(8, std::max<uint32_t>(1, ctx->tables.min_len)) + 64;
        return hpack_run_slice(ctx, encode, count, in, in_off + first, in_off[first], mode, std::min(out_capacity, room), size,
                               st);
    };
    auto finish = [&](aws_huffman_batch_ctx *ctx, size_t first, size_t count, bool last, const uint64_t *base,
                      const uint64_t *size, const uint64_t *total, cudaStream_t st) {
        return hpack_run_finish(ctx, encode, count, last, base[0], size[0], total[0], out, out_capacity, out_off + first,
                                status ? status + first : nullptr, st);
    };
    return hpack_multi(ctxs, n_ctx, n, in_off, run, finish);
}

int hpack_blocks_decode_multi(
    aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, size_t n, const uint8_t *in, const uint64_t *in_off,
    aws_hpack_header_lists *out, int32_t *status) {
    bool done;
    if (check_contexts(ctxs, n_ctx)) return AWS_OP_ERR;
    if (n_ctx == 1) return hpack_blocks_decode_host(ctxs[0], n, in, in_off, out, status);
    if (hpack_blocks_decode_args(n, in, in_off, out, &done) || done) return done ? AWS_OP_SUCCESS : AWS_OP_ERR;
    auto run = [&](aws_huffman_batch_ctx *ctx, size_t first, size_t count, uint64_t *size, cudaStream_t st) {
        // (no capacities of the shard's own: its staging is sized from its totals, the caller's decide at the finish)
        return hpack_blocks_decode_slice(ctx, count, in, in_off + first, in_off[first], ~0ull, ~0ull, size, st);
    };
    auto finish = [&](aws_huffman_batch_ctx *ctx, size_t first, size_t count, bool last, const uint64_t *base,
                      const uint64_t *size, const uint64_t *total, cudaStream_t st) {
        return hpack_blocks_decode_finish(ctx, first, count, last, base, size, total, out, status, st);
    };
    return hpack_multi(ctxs, n_ctx, n, in_off, run, finish);
}

int hpack_blocks_encode_multi(
    aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, const aws_hpack_header_lists *in, bool records, uint32_t mode,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_off, int32_t *status) {
    bool done;
    if (check_contexts(ctxs, n_ctx)) return AWS_OP_ERR;
    if (n_ctx == 1) return hpack_blocks_encode_host(ctxs[0], in, records, mode, out, out_capacity, out_off, status);
    if (hpack_blocks_encode_args(in, records, out, out_capacity, out_off, &done) || done)
        return done ? AWS_OP_SUCCESS : AWS_OP_ERR;
    // shards balanced by string octets: list i's start at string_offsets[2 * field_offsets[i]]
    const size_t n = in->n;
    std::vector<uint64_t> weight(n + 1);
    for (size_t i = 0; i <= n; ++i) weight[i] = in->string_offsets[2 * in->field_offsets[i]];
    auto run = [&](aws_huffman_batch_ctx *ctx, size_t first, size_t count, uint64_t *size, cudaStream_t st) {
        // the shard's staging holds all its output: per field a representation of at most 10 octets and two literals
        // behind prefixes of at most 10 octets each, no longer than the strings unless every literal is Huffman-coded
        const uint64_t fields = in->field_offsets[first + count] - in->field_offsets[first];
        const uint64_t octets = weight[first + count] - weight[first];
        const uint64_t expand = mode == hb::kHpackAlways ? (std::max<uint32_t>(1, ctx->tables.max_len) + 7) / 8 : 1;
        const uint64_t room = octets * expand + 30 * fields + 64;
        return hpack_blocks_encode_slice(ctx, in, first, count, records, mode, std::min(out_capacity, room), size, st);
    };
    auto finish = [&](aws_huffman_batch_ctx *ctx, size_t first, size_t count, bool last, const uint64_t *base,
                      const uint64_t *size, const uint64_t *total, cudaStream_t st) {
        return hpack_blocks_encode_finish(ctx, first, count, last, records, base[0], size[0], total[0], out, out_capacity,
                                          out_off, status, st);
    };
    return hpack_multi(ctxs, n_ctx, n, weight.data(), run, finish);
}

}  // namespace

extern "C" {

static int hb_ctx_from_codes(
    struct aws_huffman_batch_ctx **out_ctx,
    const struct aws_huffman_code *codes,
    struct aws_huffman_symbol_coder *coder, /* optional: its decode callback is cross-checked */
    uint8_t eos_padding,
    int device_id);

int aws_huffman_batch_ctx_new(
    struct aws_huffman_batch_ctx **out_ctx,
    struct aws_huffman_symbol_coder *coder,
    uint8_t eos_padding,
    int device_id) {

    if (!out_ctx || !coder || !coder->encode) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    *out_ctx = nullptr;
    // Materialise the coder once over all 256 symbols (host callbacks never run again).
    struct aws_huffman_code codes[256];
    for (int s = 0; s < 256; ++s) codes[s] = coder->encode((uint8_t)s, coder->userdata);
    return hb_ctx_from_codes(out_ctx, codes, coder, eos_padding, device_id);
}

int aws_huffman_batch_ctx_new_from_code_table(
    struct aws_huffman_batch_ctx **out_ctx,
    const struct aws_huffman_code *code_table,
    uint8_t eos_padding,
    int device_id) {

    if (!out_ctx || !code_table) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    *out_ctx = nullptr;
    return hb_ctx_from_codes(out_ctx, code_table, nullptr, eos_padding, device_id);
}

static int hb_ctx_from_codes(
    struct aws_huffman_batch_ctx **out_ctx,
    const struct aws_huffman_code *codes,
    struct aws_huffman_symbol_coder *coder,
    uint8_t eos_padding,
    int device_id) {

    uint32_t patterns[256];
    uint8_t num_bits[256];
    uint2 enc[256];
    for (int s = 0; s < 256; ++s) {
        const struct aws_huffman_code c = codes[s];
        if (c.num_bits > 32) return aws_raise_error(AWS_ERROR_COMPRESSION_INVALID_CODE_TABLE);
        const uint32_t mask = c.num_bits >= 32 ? 0xffffffffu : ((1u << c.num_bits) - 1u);
        patterns[s] = c.pattern & mask;
        num_bits[s] = c.num_bits;
        enc[s] = make_uint2(patterns[s], c.num_bits);
    }
    struct huffman_lut lut;
    const int lut_rc = huffman_lut_build(&lut, patterns, num_bits, kLutRootBits, kLutSubBits);
    if (lut_rc == HUFFMAN_LUT_ERR_OOM) return aws_raise_error(AWS_ERROR_OOM);
    if (lut_rc != HUFFMAN_LUT_OK) return aws_raise_error(AWS_ERROR_COMPRESSION_INVALID_CODE_TABLE);

    // Optional cross-check of the coder's own decode callback on every code (what the reference's
    // huffman_symbol_decoder test does, tests/huffman_test.c:199-220).
    if (coder && coder->decode) {
        for (int s = 0; s < 256; ++s) {
            if (!num_bits[s]) continue;
            uint8_t sym = 0;
            const uint8_t used = coder->decode(patterns[s] << (32 - num_bits[s]), &sym, coder->userdata);
            if (used != num_bits[s] || sym != s) {
                huffman_lut_clean_up(&lut);
                return aws_raise_error(AWS_ERROR_COMPRESSION_INVALID_CODE_TABLE);
            }
        }
    }

    aws_huffman_batch_ctx *ctx = new (std::nothrow) aws_huffman_batch_ctx();
    if (!ctx) {
        huffman_lut_clean_up(&lut);
        return aws_raise_error(AWS_ERROR_OOM);
    }
    ctx->device = device_id;

    auto fail = [&](cudaError_t err, const char *what, int line) {
        hb_note_cuda_error(err, what, line);
        huffman_lut_clean_up(&lut);
        aws_huffman_batch_ctx_destroy(ctx);
        return aws_raise_error(AWS_ERROR_COMPRESSION_DEVICE_FAILURE);
    };
#define HB_CTX_TRY(expr)                                                                                               \
    do {                                                                                                               \
        cudaError_t e_ = (expr);                                                                                       \
        if (e_ != cudaSuccess) return fail(e_, #expr, __LINE__);                                                       \
    } while (0)

    int count = 0;
    HB_CTX_TRY(cudaGetDeviceCount(&count));
    if (device_id < 0 || device_id >= count) return fail(cudaErrorInvalidDevice, "device_id", __LINE__);
    HB_CTX_TRY(cudaSetDevice(device_id));
    HB_CTX_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    HB_CTX_TRY(cudaEventCreateWithFlags(&ctx->scratch_free, cudaEventDisableTiming));
    ctx->force_generic = getenv("AWS_HUFFMAN_BATCH_FORCE_GENERIC") != nullptr;
    ctx->no_slots = getenv("AWS_HUFFMAN_BATCH_NO_SLOTS") != nullptr;
    ctx->no_strings = getenv("AWS_HUFFMAN_BATCH_NO_STRINGS") != nullptr;
    ctx->no_fused_stream = getenv("AWS_HUFFMAN_BATCH_NO_FUSED_STREAM") != nullptr;
    HB_CTX_TRY(cudaMalloc(&ctx->d_enc, sizeof(enc)));
    HB_CTX_TRY(cudaMalloc(&ctx->d_lut, (size_t)lut.count * sizeof(uint32_t)));
    HB_CTX_TRY(cudaMemcpy(ctx->d_enc, enc, sizeof(enc), cudaMemcpyHostToDevice));
    {
        // re-encode for the device (format: device_common.cuh); root entries get a second symbol when
        // two complete codes fit in the root index
        std::vector<uint32_t> dev(lut.count);
        auto single = [](uint32_t len, uint32_t sym) { return (len << 24) | (sym << 8) | (len << 2) | 1u; };
        for (uint32_t i = 0; i < lut.count; ++i) {
            const uint32_t e = lut.entries[i];
            if (e == 0) dev[i] = 0;
            else if (HUFFMAN_LUT_IS_LEAF(e)) dev[i] = single(HUFFMAN_LUT_LEAF_LEN(e), HUFFMAN_LUT_LEAF_SYMBOL(e));
            else dev[i] = (HUFFMAN_LUT_LINK_WIDTH(e) << 20) | HUFFMAN_LUT_LINK_BASE(e);
        }
        if (lut.count >= (1u << 20)) {
            huffman_lut_clean_up(&lut);
            aws_huffman_batch_ctx_destroy(ctx);
            return aws_raise_error(AWS_ERROR_COMPRESSION_INVALID_CODE_TABLE);
        }
        for (uint32_t i = 0; i < (1u << lut.root_bits); ++i) {
            const uint32_t e = lut.entries[i];
            if (!HUFFMAN_LUT_IS_LEAF(e)) continue;
            const uint32_t len1 = HUFFMAN_LUT_LEAF_LEN(e);
            if (len1 >= lut.root_bits) continue;
            const uint32_t rest = lut.root_bits - len1;  // index bits left after the first code
            const uint32_t window2 = (i << (32 - lut.root_bits)) << len1;
            uint8_t sym2 = 0;
            const uint8_t len2 = huffman_lut_decode(&lut, window2, &sym2);
            if (len2 != 0 && len2 <= rest)
                dev[i] = ((len1 + len2) << 24) | ((uint32_t)sym2 << 16) | ((uint32_t)HUFFMAN_LUT_LEAF_SYMBOL(e) << 8) |
                         (len1 << 2) | 2u;
        }
        HB_CTX_TRY(cudaMemcpy(ctx->d_lut, dev.data(), (size_t)lut.count * sizeof(uint32_t), cudaMemcpyHostToDevice));
        // LUT2 (decode_span_lean): the same tables as 64-bit entries {symbols, count | bits consumed, next table};
        // tables are 32-byte aligned (the step takes the table address and the index shift out of one word)
        std::vector<uint2> lut2;
        const uint32_t root_y = 32u - lut.root_bits;  // next step: root table (offset 0)
        lut2.resize((size_t)1 << lut.root_bits);
        while (lut2.size() & 3) lut2.push_back(uint2{0, 0});
        const uint32_t trap_base = (uint32_t)lut2.size();
        const uint32_t trap_y = (trap_base * 8u) | 31u;  // index width 1, nothing consumed: a trapped lane stays
        for (int i = 0; i < 4; ++i) lut2.push_back(uint2{0, trap_y});
        struct Conv {
            std::vector<uint2> &out;
            const std::vector<uint32_t> &dev;
            uint32_t root_y, trap_y;
            void table(uint32_t new_base, uint32_t old_base, uint32_t width, uint32_t used) {
                for (uint32_t idx = 0; idx < (1u << width); ++idx) {
                    const uint32_t e = dev[old_base + idx];
                    uint2 o;
                    if (e == 0) {
                        o = uint2{0, trap_y};
                    } else if (e >= 0x01000000u) {
                        const uint32_t total = e >> 24, len1 = (e >> 2) & 63u, cnt = e & 3u;
                        o.x = ((e >> 8) & 0xffu) | (((e >> 16) & 0xffu) << 8) | (len1 << 16) | (cnt << 30);
                        o.y = root_y | ((total - used) << 24);
                    } else {
                        const uint32_t w2 = (e >> 20) & 0xfu, b2 = e & 0xFFFFFu;
                        size_t child = (out.size() + 3) & ~size_t(3);
                        out.resize(child + std::max<size_t>(4, (size_t)1 << w2), uint2{0, trap_y});
                        table((uint32_t)child, b2, w2, used + width);
                        o.x = 0;
                        o.y = ((uint32_t)child * 8u) | (32u - w2) | (width << 24);
                    }
                    out[new_base + idx] = o;
                }
            }
        } conv{lut2, dev, root_y, trap_y};
        conv.table(0, 0, lut.root_bits, 0);
        while (lut2.size() & 3) lut2.push_back(uint2{0, trap_y});
        ctx->lut2_count = (uint32_t)lut2.size();
        ctx->lut2_trap = trap_base;
        HB_CTX_TRY(cudaMalloc(&ctx->d_lut2, lut2.size() * sizeof(uint2)));
        HB_CTX_TRY(cudaMemcpy(ctx->d_lut2, lut2.data(), lut2.size() * sizeof(uint2), cudaMemcpyHostToDevice));
    }
#undef HB_CTX_TRY

    ctx->tables.enc = ctx->d_enc;
    ctx->tables.lut = ctx->d_lut;
    ctx->tables.lut_count = lut.count;
    ctx->tables.lut_root_bits = lut.root_bits;
    ctx->tables.min_len = lut.min_len;
    ctx->tables.max_len = lut.max_len;
    ctx->tables.has_unknown = lut.has_unknown_symbols;
    ctx->tables.eos_padding = eos_padding;
    ctx->lut_smem_entries = std::min<uint32_t>(lut.count, kLutMaxSmemEntries);
    if (ctx->lut_smem_entries < (1u << lut.root_bits)) ctx->lut_smem_entries = 1u << lut.root_bits;
    huffman_lut_clean_up(&lut);
    if (configure_kernels(ctx)) {
        aws_huffman_batch_ctx_destroy(ctx);
        return AWS_OP_ERR;
    }

    *out_ctx = ctx;
    return AWS_OP_SUCCESS;
}

void aws_huffman_batch_ctx_destroy(struct aws_huffman_batch_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    delete ctx;
    (void)cudaGetLastError();
}

int aws_huffman_encode_batch(struct aws_huffman_batch_ctx *ctx, const struct aws_huffman_batch *batch) {
    return run_host_batch(ctx, batch, true);
}

int aws_huffman_decode_batch(struct aws_huffman_batch_ctx *ctx, const struct aws_huffman_batch *batch) {
    return run_host_batch(ctx, batch, false);
}

int aws_huffman_encode_batch_resume(struct aws_huffman_batch_ctx *ctx, const struct aws_huffman_batch *batch) {
    return run_host_batch(ctx, batch, true, true);
}

int aws_huffman_decode_batch_resume(struct aws_huffman_batch_ctx *ctx, const struct aws_huffman_batch *batch) {
    return run_host_batch(ctx, batch, false, true);
}

int aws_huffman_encode_batch_resume_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_huffman_batch *batch,
    void *cuda_stream) {
    return run_device_batch(ctx, batch, cuda_stream, true, true);
}

int aws_huffman_decode_batch_resume_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_huffman_batch *batch,
    void *cuda_stream) {
    return run_device_batch(ctx, batch, cuda_stream, false, true);
}

int aws_huffman_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_huffman_batch *batch,
    void *cuda_stream) {
    return run_device_batch(ctx, batch, cuda_stream, true, false);
}

int aws_huffman_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const struct aws_huffman_batch *batch,
    void *cuda_stream) {
    return run_device_batch(ctx, batch, cuda_stream, false, false);
}

int aws_huffman_histogram_device(const uint8_t *in, uint64_t size, uint64_t *counts, void *cuda_stream) {
    if (!counts || (size && !in)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return histogram_on_device(in, size, counts, static_cast<cudaStream_t>(cuda_stream));
}

int aws_huffman_histogram(int device_id, const uint8_t *in, uint64_t size, uint64_t counts[256]) {
    if (!counts || (size && !in)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    HB_CUDA_TRY(cudaSetDevice(device_id));
    uint8_t *d_in = nullptr;
    uint64_t *d_counts = nullptr;
    cudaStream_t st = nullptr;
    int rc = AWS_OP_ERR;
    do {
        if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) break;
        if (cudaMalloc(&d_counts, 256 * sizeof(uint64_t)) != cudaSuccess) break;
        if (size && cudaMalloc(&d_in, size) != cudaSuccess) break;
        if (size && cudaMemcpyAsync(d_in, in, size, cudaMemcpyHostToDevice, st) != cudaSuccess) break;
        if (histogram_on_device(d_in, size, d_counts, st)) break;
        if (cudaMemcpyAsync(counts, d_counts, 256 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st) != cudaSuccess) break;
        if (cudaStreamSynchronize(st) != cudaSuccess) break;
        rc = AWS_OP_SUCCESS;
    } while (false);
    if (d_in) cudaFree(d_in);
    if (d_counts) cudaFree(d_counts);
    if (st) cudaStreamDestroy(st);
    if (rc) {
        (void)cudaGetLastError();
        return aws_raise_error(AWS_ERROR_COMPRESSION_DEVICE_FAILURE);
    }
    return AWS_OP_SUCCESS;
}

int aws_hpack_string_encode_batch(
    struct aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets,
    enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets) {
    if ((unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return hpack_run_host(ctx, true, n, in, in_offsets, (uint32_t)mode, out, out_capacity, out_offsets, nullptr);
}

int aws_hpack_string_decode_batch(
    struct aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_offsets, int32_t *status) {
    return hpack_run_host(ctx, false, n, in, in_offsets, 0, out, out_capacity, out_offsets, status);
}

int aws_hpack_string_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets, uint64_t in_size,
    enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, void *cuda_stream) {
    if (!ctx || (n && (!in_offsets || !out_offsets)) || (unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    if (n == 0) return call_end(ctx, st, write_empty_packed(out_offsets, st));
    return call_end(
        ctx, st, hpack_encode_on_device(ctx, n, in, in_offsets, in_size, (uint32_t)mode, out, out_capacity, out_offsets, st));
}

int aws_hpack_string_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets, uint64_t in_size,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status, void *cuda_stream) {
    if (!ctx || (n && (!in_offsets || !out_offsets))) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    if (n == 0) return call_end(ctx, st, write_empty_packed(out_offsets, st));
    return call_end(
        ctx, st, hpack_decode_on_device(ctx, n, in, in_offsets, in_size, out, out_capacity, out_offsets, status, st));
}

int aws_hpack_header_block_decode_batch(
    struct aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets,
    struct aws_hpack_header_lists *out, int32_t *status) {
    return hpack_blocks_decode_host(ctx, n, in, in_offsets, out, status);
}

int aws_hpack_header_block_encode_batch(
    struct aws_huffman_batch_ctx *ctx, const struct aws_hpack_header_lists *in, enum aws_hpack_huffman_mode mode,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets) {
    if ((unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return hpack_blocks_encode_host(ctx, in, false, (uint32_t)mode, out, out_capacity, out_offsets, nullptr);
}

int aws_hpack_header_block_encode_records_batch(
    struct aws_huffman_batch_ctx *ctx, const struct aws_hpack_header_lists *in, enum aws_hpack_huffman_mode mode,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status) {
    if ((unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return hpack_blocks_encode_host(ctx, in, true, (uint32_t)mode, out, out_capacity, out_offsets, status);
}

int aws_hpack_header_block_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets, uint64_t in_size,
    struct aws_hpack_header_lists *out, int32_t *status, void *cuda_stream) {
    if (!ctx || (n && !in_offsets) || (in_size && !in) || check_block_lists(out, true) || out->n != n)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, hpack_blocks_decode_on_device(ctx, n, in, in_offsets, block_lists(out), status, false, st));
}

int aws_hpack_header_block_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx, const struct aws_hpack_header_lists *in, uint64_t num_fields,
    uint64_t strings_size, enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets,
    void *cuda_stream) {
    if (!ctx || check_block_lists(in, false) || !out_offsets || (out_capacity && !out) || (strings_size && !in->strings) ||
        (unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st,
                           hpack_blocks_encode_on_device(ctx, in->n, in->field_offsets, num_fields, in->never_indexed, nullptr,
                                                         nullptr, in->strings, in->string_offsets, strings_size, (uint32_t)mode,
                                                         out, out_capacity, out_offsets, nullptr, st));
}

int aws_hpack_header_block_encode_records_batch_device(
    struct aws_huffman_batch_ctx *ctx, const struct aws_hpack_header_lists *in, uint64_t num_fields,
    uint64_t strings_size, enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets,
    int32_t *status, void *cuda_stream) {
    if (!ctx || check_block_lists(in, false) || !in->field_kind || !in->field_index || !out_offsets ||
        (out_capacity && !out) || (strings_size && !in->strings) || (unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st,
                           hpack_blocks_encode_on_device(ctx, in->n, in->field_offsets, num_fields, in->never_indexed,
                                                         in->field_kind, in->field_index, in->strings, in->string_offsets,
                                                         strings_size, (uint32_t)mode, out, out_capacity, out_offsets, status,
                                                         st));
}

int aws_qpack_field_section_decode_batch(
    struct aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets,
    struct aws_qpack_field_sections *out, int32_t *status) {
    return qpack_sections_decode_host(ctx, n, in, in_offsets, out, status);
}

int aws_qpack_field_section_encode_batch(
    struct aws_huffman_batch_ctx *ctx, const struct aws_qpack_field_sections *in, enum aws_hpack_huffman_mode mode,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets) {
    return qpack_sections_encode_host(ctx, in, false, (uint32_t)mode, out, out_capacity, out_offsets, nullptr);
}

int aws_qpack_field_section_encode_records_batch(
    struct aws_huffman_batch_ctx *ctx, const struct aws_qpack_field_sections *in, enum aws_hpack_huffman_mode mode,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status) {
    return qpack_sections_encode_host(ctx, in, true, (uint32_t)mode, out, out_capacity, out_offsets, status);
}

int aws_qpack_field_section_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets, uint64_t in_size,
    struct aws_qpack_field_sections *out, int32_t *status, void *cuda_stream) {
    if (!ctx || (n && !in_offsets) || (in_size && !in) || check_section_lists(out, true, false) || out->n != n)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, qpack_sections_decode_on_device(ctx, n, in, in_offsets, *out, status, false, st));
}

int aws_qpack_field_section_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx, const struct aws_qpack_field_sections *in, uint64_t num_fields,
    uint64_t strings_size, enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets,
    void *cuda_stream) {
    if (!ctx || check_section_lists(in, false, false) || !out_offsets || (out_capacity && !out) ||
        (strings_size && !in->strings) || (unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st,
                    qpack_sections_encode_on_device(ctx, in->n, in->field_offsets, num_fields, in->never_indexed, nullptr,
                                                    nullptr, nullptr, nullptr, nullptr, in->strings, in->string_offsets,
                                                    strings_size, (uint32_t)mode, out, out_capacity, out_offsets, nullptr,
                                                    st));
}

int aws_qpack_field_section_encode_records_batch_device(
    struct aws_huffman_batch_ctx *ctx, const struct aws_qpack_field_sections *in, uint64_t num_fields,
    uint64_t strings_size, enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets,
    int32_t *status, void *cuda_stream) {
    if (!ctx || check_section_lists(in, false, true) || !out_offsets || (out_capacity && !out) ||
        (strings_size && !in->strings) || (unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st,
                    qpack_sections_encode_on_device(ctx, in->n, in->field_offsets, num_fields, in->never_indexed,
                                                    in->field_kind, in->field_index, in->encoded_insert_count,
                                                    in->base_sign, in->delta_base, in->strings, in->string_offsets,
                                                    strings_size, (uint32_t)mode, out, out_capacity, out_offsets, status,
                                                    st));
}

int aws_qpack_instruction_decode_batch(
    struct aws_huffman_batch_ctx *ctx, enum aws_qpack_instruction_stream which, size_t n, const uint8_t *in,
    const uint64_t *in_offsets, struct aws_qpack_instructions *out, uint64_t *consumed, int32_t *status) {
    return qpack_instructions_decode_host(ctx, (uint32_t)which, n, in, in_offsets, out, consumed, status);
}

int aws_qpack_instruction_encode_batch(
    struct aws_huffman_batch_ctx *ctx, enum aws_qpack_instruction_stream which, const struct aws_qpack_instructions *in,
    enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status) {
    return qpack_instructions_encode_host(ctx, (uint32_t)which, in, (uint32_t)mode, out, out_capacity, out_offsets, status);
}

int aws_qpack_instruction_decode_batch_device(
    struct aws_huffman_batch_ctx *ctx, enum aws_qpack_instruction_stream which, size_t n, const uint8_t *in,
    const uint64_t *in_offsets, uint64_t in_size, struct aws_qpack_instructions *out, uint64_t *consumed, int32_t *status,
    void *cuda_stream) {
    if (!ctx || (n && (!in_offsets || !consumed)) || (in_size && !in) || check_instruction_lists(out, (uint32_t)which, true) ||
        out->n != n)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, qpack_instructions_decode_on_device(ctx, (uint32_t)which, n, in, in_offsets, *out, consumed,
                                                                 status, false, st));
}

int aws_qpack_instruction_encode_batch_device(
    struct aws_huffman_batch_ctx *ctx, enum aws_qpack_instruction_stream which, const struct aws_qpack_instructions *in,
    uint64_t num_instructions, uint64_t strings_size, enum aws_hpack_huffman_mode mode, uint8_t *out,
    uint64_t out_capacity, uint64_t *out_offsets, int32_t *status, void *cuda_stream) {
    if (!ctx || check_instruction_lists(in, (uint32_t)which, false) || !out_offsets || (out_capacity && !out) ||
        (which == AWS_QPACK_ENCODER_STREAM && strings_size && !in->strings) ||
        (unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS)
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st,
                    qpack_instructions_encode_on_device(ctx, (uint32_t)which, in->n, in->instruction_offsets,
                                                        num_instructions, in->kind, in->index, in->strings,
                                                        in->string_offsets, which == AWS_QPACK_ENCODER_STREAM ? strings_size : 0,
                                                        (uint32_t)mode, out, out_capacity, out_offsets, status, st));
}

int aws_huffman_get_encoded_length_batch(
    struct aws_huffman_batch_ctx *ctx,
    const uint8_t *in,
    const uint64_t *in_offsets,
    size_t n,
    uint64_t *lens) {
    if (!ctx || (n && (!in_offsets || !lens))) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (n == 0) return AWS_OP_SUCCESS;
    if (in_offsets[n] && !in) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    cudaStream_t st;
    if (call_begin(ctx, nullptr, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, encoded_lengths_staged(ctx, in, in_offsets, n, lens, st));
}

int aws_huffman_batch_ctx_synchronize(struct aws_huffman_batch_ctx *ctx) {
    if (!ctx) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    HB_CUDA_TRY(cudaSetDevice(ctx->device));
    HB_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return AWS_OP_SUCCESS;
}

void *aws_huffman_batch_ctx_stream(struct aws_huffman_batch_ctx *ctx) {
    return ctx ? ctx->stream : nullptr;
}

int aws_huffman_batch_ctx_device(struct aws_huffman_batch_ctx *ctx) {
    return ctx ? ctx->device : -1;
}

uint64_t aws_huffman_batch_ctx_launch_count(struct aws_huffman_batch_ctx *ctx) {
    return ctx ? ctx->launches : 0;
}

int aws_huffman_batch_plan_shards(const uint64_t *in_offsets, size_t n, size_t num_shards, size_t *shard_begin) {
    if (!shard_begin || num_shards == 0 || (n && !in_offsets)) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    const uint64_t base = n ? in_offsets[0] : 0;
    const uint64_t total = n ? in_offsets[n] - base : 0;
    shard_begin[0] = 0;
    for (size_t s = 1; s < num_shards; ++s) {
        // first item whose start offset reaches the s-th equal share of the bytes
        const uint64_t target = base + (uint64_t)(((unsigned __int128)total * s) / num_shards);
        const uint64_t *it = std::lower_bound(in_offsets, in_offsets + n, target);
        size_t idx = (size_t)(it - in_offsets);
        if (total == 0) idx = (size_t)(((unsigned __int128)n * s) / num_shards);  // all items empty: split by count
        shard_begin[s] = std::max(idx, shard_begin[s - 1]);
    }
    shard_begin[num_shards] = n;
    return AWS_OP_SUCCESS;
}

int aws_huffman_batch_concat_offsets(
    const uint64_t *const *shard_offsets,
    const size_t *shard_items,
    size_t num_shards,
    uint64_t *global_offsets) {
    if (!global_offsets || (num_shards && (!shard_offsets || !shard_items)))
        return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    uint64_t base = 0;
    size_t at = 0;
    for (size_t s = 0; s < num_shards; ++s) {
        const uint64_t *local = shard_offsets[s];
        for (size_t i = 0; i < shard_items[s]; ++i) global_offsets[at++] = base + local[i];
        if (shard_items[s]) base += local[shard_items[s]];
    }
    global_offsets[at] = base;
    return AWS_OP_SUCCESS;
}

// One batch over several contexts (one per GPU of the box, or several on one GPU): plan by bytes, one host thread
// per context drives its shard through that context's own (pipelined) host path into a private buffer, and the
// host concatenates payloads and offsets. No collective: the shards never talk to each other.
static int hb_run_multi(struct aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, const struct aws_huffman_batch *b, bool encode) {
    if (check_contexts(ctxs, n_ctx) || check_batch(b)) return AWS_OP_ERR;
    if (b->out_caps) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);  // packed layout only
    const size_t n = b->n;
    if (n == 0) {
        if (b->out_offsets) b->out_offsets[0] = 0;
        return AWS_OP_SUCCESS;
    }
    if (n_ctx == 1) return encode ? aws_huffman_encode_batch(ctxs[0], b) : aws_huffman_decode_batch(ctxs[0], b);
    std::vector<size_t> begin(n_ctx + 1);
    if (aws_huffman_batch_plan_shards(b->in_offsets, n, n_ctx, begin.data())) return AWS_OP_ERR;
    struct Shard {
        std::vector<uint64_t> in_off, out_off;
        std::vector<uint8_t> out;
    };
    std::vector<Shard> shards(n_ctx);
    if (run_shards(n_ctx, [&](size_t d) -> int {
            Shard &sh = shards[d];
            const size_t a = begin[d], nd = begin[d + 1] - a;
            if (nd == 0) return AWS_OP_SUCCESS;
            const uint64_t in0 = b->in_offsets[a], bytes_in = b->in_offsets[a + nd] - in0;
            const uint32_t max_len = std::max<uint32_t>(1, ctxs[d]->tables.max_len), min_len = std::max<uint32_t>(1, ctxs[d]->tables.min_len);
            const uint64_t room = (encode ? bytes_in * ((max_len + 7) / 8) : (bytes_in * 8) / min_len) + 64;
            sh.in_off.resize(nd + 1);
            for (size_t i = 0; i <= nd; ++i) sh.in_off[i] = b->in_offsets[a + i] - in0;
            sh.out_off.assign(nd + 1, 0);
            sh.out.resize(room);
            aws_huffman_batch sb = *b;
            sb.n = nd;
            sb.in = b->in + in0;
            sb.in_offsets = sh.in_off.data();
            sb.in_size = bytes_in;
            sb.out = sh.out.data();
            sb.out_capacity = room;
            sb.out_offsets = sh.out_off.data();
            if (b->out_lens) sb.out_lens = b->out_lens + a;
            if (b->status) sb.status = b->status + a;
            if (b->consumed) sb.consumed = b->consumed + a;
            if (b->overflow_pattern) sb.overflow_pattern = b->overflow_pattern + a;
            if (b->overflow_num_bits) sb.overflow_num_bits = b->overflow_num_bits + a;
            if (b->leftover_working_bits) sb.leftover_working_bits = b->leftover_working_bits + a;
            if (b->leftover_num_bits) sb.leftover_num_bits = b->leftover_num_bits + a;
            return encode ? aws_huffman_encode_batch(ctxs[d], &sb) : aws_huffman_decode_batch(ctxs[d], &sb);
        }))
        return AWS_OP_ERR;
    // the concatenation step
    std::vector<const uint64_t *> ptrs(n_ctx);
    std::vector<size_t> items(n_ctx);
    for (size_t d = 0; d < n_ctx; ++d) {
        items[d] = begin[d + 1] - begin[d];
        static const uint64_t zero = 0;
        ptrs[d] = items[d] ? shards[d].out_off.data() : &zero;
    }
    if (aws_huffman_batch_concat_offsets(ptrs.data(), items.data(), n_ctx, b->out_offsets)) return AWS_OP_ERR;
    if (b->out_offsets[n] > b->out_capacity) return aws_raise_error(AWS_ERROR_SHORT_BUFFER);
    for (size_t d = 0; d < n_ctx; ++d)
        if (items[d]) memcpy(b->out + b->out_offsets[begin[d]], shards[d].out.data(), (size_t)shards[d].out_off[items[d]]);
    return AWS_OP_SUCCESS;
}

int aws_huffman_encode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, const struct aws_huffman_batch *batch) {
    return hb_run_multi(ctxs, n_ctx, batch, true);
}

int aws_huffman_decode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, const struct aws_huffman_batch *batch) {
    return hb_run_multi(ctxs, n_ctx, batch, false);
}

int aws_hpack_string_encode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets,
    enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets) {
    if ((unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return hpack_literals_multi(ctxs, n_ctx, true, n, in, in_offsets, (uint32_t)mode, out, out_capacity, out_offsets, nullptr);
}

int aws_hpack_string_decode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets,
    uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status) {
    return hpack_literals_multi(ctxs, n_ctx, false, n, in, in_offsets, 0, out, out_capacity, out_offsets, status);
}

int aws_hpack_header_block_decode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, size_t n, const uint8_t *in, const uint64_t *in_offsets,
    struct aws_hpack_header_lists *out, int32_t *status) {
    return hpack_blocks_decode_multi(ctxs, n_ctx, n, in, in_offsets, out, status);
}

int aws_hpack_header_block_encode_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, const struct aws_hpack_header_lists *in,
    enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets) {
    if ((unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return hpack_blocks_encode_multi(ctxs, n_ctx, in, false, (uint32_t)mode, out, out_capacity, out_offsets, nullptr);
}

int aws_hpack_header_block_encode_records_batch_multi(
    struct aws_huffman_batch_ctx *const *ctxs, size_t n_ctx, const struct aws_hpack_header_lists *in,
    enum aws_hpack_huffman_mode mode, uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status) {
    if ((unsigned)mode > (unsigned)AWS_HPACK_HUFFMAN_ALWAYS) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    return hpack_blocks_encode_multi(ctxs, n_ctx, in, true, (uint32_t)mode, out, out_capacity, out_offsets, status);
}

int aws_huffman_get_encoded_length_batch_device(
    struct aws_huffman_batch_ctx *ctx,
    const uint8_t *in,
    const uint64_t *in_offsets,
    size_t n,
    uint64_t *lens,
    void *cuda_stream) {
    if (!ctx || (n && (!in_offsets || !lens))) return aws_raise_error(AWS_ERROR_INVALID_ARGUMENT);
    if (n == 0) return AWS_OP_SUCCESS;
    cudaStream_t st;
    if (call_begin(ctx, cuda_stream, &st)) return AWS_OP_ERR;
    return call_end(ctx, st, encoded_lengths_on_device(ctx, in, in_offsets, n, lens, st));
}

}  // extern "C"

#ifdef HB_PHASE_TIMING
// development builds only (tools/phase_probe.py): cycles per phase of decode_batch_kernel, summed over blocks
extern "C" int aws_huffman_batch_debug_phase_cycles(unsigned long long *out16, int reset) {
    if (cudaMemcpyFromSymbol(out16, hb::hb_phase_cycles, 16 * sizeof(unsigned long long)) != cudaSuccess) return -1;
    if (reset) {
        unsigned long long zero[16] = {0};
        if (cudaMemcpyToSymbol(hb::hb_phase_cycles, zero, sizeof(zero)) != cudaSuccess) return -1;
    }
    return 0;
}
extern "C" int aws_huffman_batch_debug_tile_times(unsigned long long *out /* 4 x 8192 */) {
    return cudaMemcpyFromSymbol(out, hb::hb_tile_times, sizeof(unsigned long long) * 4 * 8192) == cudaSuccess ? 0 : -1;
}
#endif
