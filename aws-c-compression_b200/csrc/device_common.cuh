// Shared device-side definitions for the batched Huffman codec (sm_100a).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace hb {

#ifdef HB_PHASE_TIMING
__device__ unsigned long long hb_phase_cycles[16];  // (development builds: tools/phase_probe.py)
__device__ unsigned long long hb_tile_times[4][8192];  // per tile: ticket, publish, resolve start, resolve end (globaltimer ns)
__device__ __forceinline__ unsigned long long hb_now_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

// Error values written to per-item status arrays (match aws-c-common / compression.h).
constexpr int32_t kStatusOk = 0;
constexpr int32_t kStatusShortBuffer = 4;       // AWS_ERROR_SHORT_BUFFER
constexpr int32_t kStatusUnknownSymbol = 3072;  // AWS_ERROR_COMPRESSION_UNKNOWN_SYMBOL

constexpr uint64_t kNoCap = ~0ull;  // "all the room it needs" (packed layout)

// Device decode LUT entry (host/huffman_lut.h entries are re-encoded at context creation):
//   leaf : [31:24] bits consumed by the whole entry (1..32)   [23:16] symbol 2   [15:8] symbol 1
//          [7:2] length of symbol 1's code   [1:0] symbols in the entry (1 or 2)
//          Root entries hold TWO symbols whenever two complete codes fit in the root index; sub-table
//          entries always hold one.
//   link : [31:24] = 0, [23:20] index width of the sub-table (1..8), [19:0] its first entry
//   hole : 0
__device__ __forceinline__ bool dlut_is_leaf(uint32_t e) { return e >= 0x01000000u; }
__device__ __forceinline__ uint32_t dlut_total_len(uint32_t e) { return e >> 24; }
__device__ __forceinline__ uint32_t dlut_len1(uint32_t e) { return (e >> 2) & 63u; }
__device__ __forceinline__ uint32_t dlut_sym1(uint32_t e) { return (e >> 8) & 0xffu; }
__device__ __forceinline__ uint32_t dlut_count(uint32_t e) { return e & 3u; }
__device__ __forceinline__ uint32_t dlut_link_width(uint32_t e) { return (e >> 20) & 0xfu; }
__device__ __forceinline__ uint32_t dlut_link_base(uint32_t e) { return e & 0xFFFFFu; }

// Device-resident tables of one context. Pointers are device pointers.
struct DeviceTables {
    const uint2 *enc;          // [256] {x = pattern (masked to num_bits), y = num_bits}
    const uint32_t *lut;       // multi-level decode LUT, `lut_count` entries
    uint32_t lut_count;
    uint32_t lut_root_bits;
    uint32_t min_len;          // shortest code length (>= 1 when the table is not empty)
    uint32_t max_len;
    uint32_t has_unknown;      // some symbol has no code
    uint32_t eos_padding;
};

// Per-call view of an aws_huffman_batch (device pointers), shared by encode and decode kernels.
struct BatchView {
    uint64_t n;
    const uint8_t *in;
    const uint64_t *in_offsets;
    uint8_t *out;
    uint64_t out_capacity;
    uint64_t *out_offsets;      // packed: produced by the scan; slotted: given
    const uint64_t *out_caps;   // nullptr = packed
    uint64_t *out_lens;         // never null inside the library (scratch when the caller passes NULL)
    int32_t *status;            // optional
    uint64_t *consumed;         // optional
    uint32_t *overflow_pattern; // encode, optional
    uint8_t *overflow_num_bits; // encode, optional
    uint64_t *leftover_working_bits;  // decode, optional
    uint8_t *leftover_num_bits;       // decode, optional
    // *_resume entry points: the encoder's overflow bits / the decoder's bit register of the PREVIOUS call are
    // read from the state arrays above (which are then required) before the new state is written to them
    bool resume;
};

__device__ __forceinline__ uint32_t lane_id() {
    return threadIdx.x & 31u;
}

__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_relaxed_u64(uint64_t *p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Warp-inclusive scan of 32-bit values.
__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v) {
    const uint32_t lane = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t up = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= (uint32_t)d) v += up;
    }
    return v;
}

__device__ __forceinline__ uint64_t warp_inclusive_scan64(uint64_t v) {
    const uint32_t lane = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint64_t up = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= (uint32_t)d) v += up;
    }
    return v;
}

// ---------------------------------------------------------------------------------------------
// Single-pass decoupled look-back (Merrill & Garland) over 64-bit sums.
// One descriptor word per tile: [63:62] flag, [61:0] value.
// ---------------------------------------------------------------------------------------------
constexpr uint64_t kLbFlagShift = 62;
constexpr uint64_t kLbValueMask = (1ull << 62) - 1;
constexpr uint64_t kLbInvalid = 0;
constexpr uint64_t kLbAggregate = 1;
constexpr uint64_t kLbPrefix = 2;

// Called by ONE FULL WARP of the tile's block. Publishes this tile's aggregate, walks back over
// predecessors, publishes the inclusive prefix and returns the exclusive prefix to every lane.
__device__ __forceinline__ uint64_t lookback_exclusive_prefix(uint64_t *tile_state, uint32_t tile, uint64_t aggregate) {
    const uint32_t lane = lane_id();
    if (tile == 0) {
        if (lane == 0) st_relaxed_u64(&tile_state[0], (kLbPrefix << kLbFlagShift) | (aggregate & kLbValueMask));
        return 0;
    }
    if (lane == 0) st_relaxed_u64(&tile_state[tile], (kLbAggregate << kLbFlagShift) | (aggregate & kLbValueMask));

    uint64_t exclusive = 0;
    int64_t look = (int64_t)tile - 1;  // highest predecessor of the current window
    while (true) {
        const int64_t idx = look - (int64_t)lane;
        uint64_t word = (kLbPrefix << kLbFlagShift);  // lanes past tile 0 act as "prefix 0"
        if (idx >= 0) {
            while (true) {
                word = ld_relaxed_u64(&tile_state[idx]);
                if ((word >> kLbFlagShift) != kLbInvalid) break;
                __nanosleep(20);
            }
        }
        const uint32_t is_prefix = (word >> kLbFlagShift) == kLbPrefix;
        const uint32_t prefix_mask = __ballot_sync(0xffffffffu, is_prefix);
        // lanes at or below the first prefix lane contribute
        const uint32_t first = prefix_mask ? (uint32_t)(__ffs(prefix_mask) - 1) : 32u;
        uint64_t contrib = (lane <= first) ? (word & kLbValueMask) : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, d);
        exclusive += contrib;
        if (prefix_mask) break;
        look -= 32;
    }
    if (lane == 0)
        st_relaxed_u64(&tile_state[tile], (kLbPrefix << kLbFlagShift) | ((exclusive + aggregate) & kLbValueMask));
    return exclusive;
}

// The same look-back in two halves, for kernels that want slack between them (the single-pass decoders
// publish a tile's aggregate at once and resolve its prefix ONE TILE LATER, so no block ever stands still
// waiting for a slower predecessor).
// One thread, as early as possible:
__device__ __forceinline__ void lookback_publish_aggregate(uint64_t *tile_state, uint32_t tile, uint64_t aggregate) {
    const uint64_t flag = tile == 0 ? kLbPrefix : kLbAggregate;
    st_relaxed_u64(&tile_state[tile], (flag << kLbFlagShift) | (aggregate & kLbValueMask));
}
// One full warp, any time later: returns the exclusive prefix of `tile` to every lane and publishes the
// inclusive one. A round is ONE 256-bit strong load per lane (4 descriptors, 128 per round; strong loads of
// a warp are served one after the other, see encode_tiled.cuh); lane 0 holds the closest group. A window
// whose closest descriptors are not published yet is read again as a whole after a short sleep.
// tile_state must be 32-byte aligned.
__device__ __forceinline__ uint64_t lookback_resolve(uint64_t *tile_state, uint32_t tile, uint64_t aggregate) {
    const uint32_t lane = lane_id();
    if (tile == 0) return 0;
#ifdef HB_ABL_NO_LOOKBACK  // (timing-only ablation: wrong output positions)
    return 0;
#endif
    uint64_t exclusive = 0;
    int64_t gtop = ((int64_t)tile - 1) >> 2;  // closest group of four descriptors
    uint32_t rtop = (tile - 1) & 3;           // last element of that group that is a predecessor
    while (true) {
        const int64_t g = gtop - (int64_t)lane;
        uint64_t word[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) word[e] = kLbPrefix << kLbFlagShift;  // "tile -1": prefix 0
        if (g >= 0)
            asm volatile("ld.relaxed.gpu.global.v4.b64 {%0, %1, %2, %3}, [%4];"
                         : "=l"(word[0]), "=l"(word[1]), "=l"(word[2]), "=l"(word[3])
                         : "l"(tile_state + 4 * g)
                         : "memory");
        const uint32_t last = lane == 0 ? rtop : 3u;
        // walk my group from the closest element back: sum aggregates up to and including the first prefix
        uint64_t sum = 0;
        bool found = false, missing = false;
#pragma unroll
        for (int e = 3; e >= 0; --e) {
            if ((uint32_t)e <= last && !found && !missing) {
                const uint64_t status = word[e] >> kLbFlagShift;
                if (status == kLbInvalid) {
                    missing = true;
                } else {
                    sum += word[e] & kLbValueMask;
                    found = status == kLbPrefix;
                }
            }
        }
        const uint32_t pmask = __ballot_sync(0xffffffffu, found);
        const uint32_t first = pmask ? (uint32_t)(__ffs(pmask) - 1) : 32u;
        if (__any_sync(0xffffffffu, missing && lane <= first)) {
#ifdef HB_PHASE_TIMING
            if (lane == 0) atomicAdd(&hb_phase_cycles[9], 1ull);
#endif
            __nanosleep(100);
            continue;
        }
#ifdef HB_PHASE_TIMING
        if (lane == 0) atomicAdd(&hb_phase_cycles[10], 1ull);
#endif
        uint64_t contrib = lane <= first ? sum : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, d);
        exclusive += contrib;
        if (pmask) break;
        gtop -= 32;
        rtop = 3;
    }
    if (lane == 0)
        st_relaxed_u64(&tile_state[tile], (kLbPrefix << kLbFlagShift) | ((exclusive + aggregate) & kLbValueMask));
    return exclusive;
}

// One full warp: the exclusive prefix of `tile` alone — the sum over its predecessors, which does not depend on
// the tile's own aggregate, so it can be started as soon as the tile is TAKEN and runs next to the tile's own work.
// Nothing is published (the caller stores the inclusive prefix once it knows both halves).
__device__ __forceinline__ uint64_t lookback_exclusive(uint64_t *tile_state, uint32_t tile) {
    const uint32_t lane = lane_id();
    if (tile == 0) return 0;
    uint64_t exclusive = 0;
    int64_t gtop = ((int64_t)tile - 1) >> 2;
    uint32_t rtop = (tile - 1) & 3;
    while (true) {
        const int64_t g = gtop - (int64_t)lane;
        uint64_t word[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) word[e] = kLbPrefix << kLbFlagShift;
        if (g >= 0)
            asm volatile("ld.relaxed.gpu.global.v4.b64 {%0, %1, %2, %3}, [%4];"
                         : "=l"(word[0]), "=l"(word[1]), "=l"(word[2]), "=l"(word[3])
                         : "l"(tile_state + 4 * g)
                         : "memory");
        const uint32_t last = lane == 0 ? rtop : 3u;
        uint64_t sum = 0;
        bool found = false, missing = false;
#pragma unroll
        for (int e = 3; e >= 0; --e) {
            if ((uint32_t)e <= last && !found && !missing) {
                const uint64_t status = word[e] >> kLbFlagShift;
                if (status == kLbInvalid) {
                    missing = true;
                } else {
                    sum += word[e] & kLbValueMask;
                    found = status == kLbPrefix;
                }
            }
        }
        const uint32_t pmask = __ballot_sync(0xffffffffu, found);
        const uint32_t first = pmask ? (uint32_t)(__ffs(pmask) - 1) : 32u;
        if (__any_sync(0xffffffffu, missing && lane <= first)) {
            __nanosleep(400);  // (the predecessors are still decoding: this runs next to the tile's own work)
            continue;
        }
        uint64_t contrib = lane <= first ? sum : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, d);
        exclusive += contrib;
        if (pmask) break;
        gtop -= 32;
        rtop = 3;
    }
    return exclusive;
}

}  // namespace hb
