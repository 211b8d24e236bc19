// UTF-8 ingest (sm_100a): log files are UTF-8 on disk (the reference reads its definitions that way,
// io/InputLineReader.java:51; callers of Gorp.extract hold the decoded Strings). gorp_extract_text_utf8 ships the BYTES
// over PCIe — one byte per ASCII character instead of two — and decodes them to UTF-16 on the device, which is what
// `new String(bytes, UTF_8)` would have produced on the host; the result offsets are UTF-16 units of that decoded text.
//
//   pass 1  utf8_count   per 4096-byte tile: UTF-16 units its bytes start (0 for a continuation byte, 2 for a 4-byte lead,
//                        else 1) + validation of every sequence (Unicode table 3-7: no overlongs, no surrogates, <= U+10FFFF,
//                        no truncated sequence); the first malformed byte offset is reported (atomicMin)
//           scan         exclusive prefix of the tile counts (scan_u32_to_i64)
//   pass 2  utf8_write   block scan inside the tile, every thread decodes the sequences that START in its 16 bytes
// Both passes are plain HBM streams (1 byte read per unit in pass 1, 1 byte read + 2 bytes written in pass 2).
//
// gorp_extract_text_utf8_bytes gives the same results in byte coordinates of the caller's buffer: a byte '\n' index of
// the piece (utf8_nl_count_mask_kernel + K1's scatter) and a gather that converts the unit rows (utf8_rows_kernel).
//
// gorp_extract_lines_utf8 (strings as UTF-8 bytes + offsets): pass 1 also leaves a unit prefix per 16-byte slice, then
// utf8_line_units_kernel turns each string's byte offset into its unit offset and checks that no string boundary cuts a
// sequence; after pass 2 the lines form of the pipeline runs on the decoded piece and utf8_rows_kernel<true> maps its rows
// back to the caller's bytes.
#include "device_common.cuh"

namespace gorp {

namespace {

constexpr int kUtf8Threads = 256;
constexpr int kUtf8PerThread = 16;
constexpr int kUtf8Tile = kUtf8Threads * kUtf8PerThread;

__device__ __forceinline__ uint32_t byte_at(const uint8_t* __restrict__ src, int64_t i, int64_t n) {
    return i < n ? static_cast<uint32_t>(__ldg(src + i)) : 0x100u;  // 0x100: "no byte" (never a continuation byte)
}

// 0x01 per byte of w whose __vcmp*4 result byte is 0xFF, packed to bits 0..3
__device__ __forceinline__ uint32_t byte_bits(uint32_t m) {
    return ((m >> 7) & 1u) | ((m >> 14) & 2u) | ((m >> 21) & 4u) | ((m >> 28) & 8u);
}

// length of the well-formed sequence that starts with lead byte b0 at position i (1..4), or 0 when malformed
__device__ __forceinline__ uint32_t sequence_length(const uint8_t* __restrict__ src, int64_t i, int64_t n, uint32_t b0) {
    if (b0 < 0x80u) return 1;
    if (b0 < 0xC2u) return 0;  // continuation byte in lead position, or an overlong 2-byte lead (C0, C1)
    const uint32_t b1 = byte_at(src, i + 1, n);
    if (b0 < 0xE0u) return (b1 & 0xC0u) == 0x80u && b1 < 0x100u ? 2u : 0u;
    const uint32_t b2 = byte_at(src, i + 2, n);
    if (b0 < 0xF0u) {
        const uint32_t lo = b0 == 0xE0u ? 0xA0u : 0x80u, hi = b0 == 0xEDu ? 0x9Fu : 0xBFu;  // no overlongs, no surrogates
        return b1 >= lo && b1 <= hi && (b2 & 0xC0u) == 0x80u && b2 < 0x100u ? 3u : 0u;
    }
    if (b0 > 0xF4u) return 0;
    const uint32_t b3 = byte_at(src, i + 3, n);
    const uint32_t lo = b0 == 0xF0u ? 0x90u : 0x80u, hi = b0 == 0xF4u ? 0x8Fu : 0xBFu;  // U+10000 .. U+10FFFF
    return b1 >= lo && b1 <= hi && (b2 & 0xC0u) == 0x80u && b2 < 0x100u && (b3 & 0xC0u) == 0x80u && b3 < 0x100u ? 4u : 0u;
}

__device__ __forceinline__ uint32_t block_sum(uint32_t v, uint32_t* s_warp) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
    __syncthreads();
    uint32_t t = 0;
    for (int w = 0; w < kUtf8Threads / 32; ++w) t += s_warp[w];
    __syncthreads();
    return t;
}

// kLines (gorp_extract_lines_utf8): also writes slice_units[i] = units of the tile before the 16-byte slice i (exclusive,
// tile-relative: < 4096, a u16), so that a string's unit offset is one lookup away (utf8_line_units_kernel).
template <bool kLines>
__global__ void __launch_bounds__(kUtf8Threads) utf8_count_kernel(const uint8_t* __restrict__ src, int64_t n, uint32_t* __restrict__ tile_counts,
                                                                 unsigned long long* __restrict__ first_bad, uint16_t* __restrict__ slice_units) {
    __shared__ uint32_t s_warp[kUtf8Threads / 32];
    const int64_t n_tiles = (n + kUtf8Tile - 1) / kUtf8Tile;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t p0 = tile * kUtf8Tile + static_cast<int64_t>(threadIdx.x) * kUtf8PerThread;
        uint32_t units = 0;
        if (p0 < n) {
            __align__(16) uint8_t b[kUtf8PerThread];
            if (p0 + kUtf8PerThread <= n) {
                *reinterpret_cast<uint4*>(b) = __ldg(reinterpret_cast<const uint4*>(src + p0));
            } else {
                for (int k = 0; k < kUtf8PerThread; ++k) b[k] = p0 + k < n ? __ldg(src + p0 + k) : 0x80;  // padding: counts nothing
            }
            // a continuation byte is legal only inside a sequence: the lead that owns it is checked by the thread that holds
            // the lead, so here every NON-continuation byte is validated as the start of a sequence, and a continuation byte
            // must be covered by the sequence that precedes it (checked by walking the sequences of this thread's range)
            int64_t expect_until = p0;  // continuation bytes before this position belong to a sequence begun earlier
            {   // how far does a sequence begun before p0 reach? look back up to 3 bytes for its lead
                for (int back = 1; back <= 3 && p0 - back >= 0; ++back) {
                    const uint32_t pb = __ldg(src + p0 - back);
                    if ((pb & 0xC0u) != 0x80u) {
                        const uint32_t len = sequence_length(src, p0 - back, n, pb);
                        if (len > static_cast<uint32_t>(back)) expect_until = p0 - back + len;
                        break;
                    }
                }
            }
            for (int k = 0; k < kUtf8PerThread; ++k) {
                const int64_t p = p0 + k;
                if (p >= n) break;
                const uint32_t c = b[k];
                if ((c & 0xC0u) == 0x80u) {
                    if (p >= expect_until) atomicMin(first_bad, static_cast<unsigned long long>(p));  // stray continuation byte
                    continue;
                }
                if (p < expect_until) {  // a lead byte inside an unfinished sequence (the lead's own check reports it)
                    continue;
                }
                const uint32_t len = sequence_length(src, p, n, c);
                if (len == 0) atomicMin(first_bad, static_cast<unsigned long long>(p));
                expect_until = p + (len ? len : 1);
                units += c >= 0xF0u ? 2u : 1u;
            }
        }
        if constexpr (kLines) {
            const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
            uint32_t incl = units;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= static_cast<uint32_t>(o)) incl += t;
            }
            if (lane == 31) s_warp[warp] = incl;
            __syncthreads();
            uint32_t before = 0, total = 0;
            for (uint32_t w = 0; w < kUtf8Threads / 32; ++w) {
                before += w < warp ? s_warp[w] : 0u;
                total += s_warp[w];
            }
            __syncthreads();
            if (p0 < n) slice_units[p0 / kUtf8PerThread] = static_cast<uint16_t>(before + incl - units);
            if (threadIdx.x == 0) tile_counts[tile] = total;
        } else {
            const uint32_t total = block_sum(units, s_warp);
            if (threadIdx.x == 0) tile_counts[tile] = total;
        }
    }
}

// Unit offsets of the strings of one piece (gorp_extract_lines_utf8), one thread per offset: byte offset b (relative to the
// piece) -> tile_base[b / 4096] + slice_units[b / 16] + units of bytes [b & ~15, b) (one 16-byte load), O(1) per string.
// It also checks the boundaries the count pass cannot see: a string that ends inside a sequence the next string completes
// (the concatenation is well-formed, the strings are not). For an interior offset b whose byte is a continuation byte, the
// string before b fails at the lead p of the cut sequence (p in [b - 3, b), the sequence reaching past b); with no such lead,
// the string that starts at b fails at b. The lowest offending byte goes to first_bad (atomicMin, as the count pass).
// order_bad (offsets that come from device memory, gorp_extract_lines_utf8_device; nullptr when the host checked them): the
// lowest i with byte_off[i + 1] < byte_off[i] (atomicMin), the index the host check reports. An offset outside
// [base, base + n] is never dereferenced (its unit offset is left 0); such an offset implies a decreasing pair, so the
// call fails on order_bad before anything reads unit_off.
__global__ void __launch_bounds__(kUtf8Threads) utf8_line_units_kernel(const uint8_t* __restrict__ src, int64_t n, const int64_t* __restrict__ byte_off,
                                                                      int64_t n_off, int64_t base, const int64_t* __restrict__ tile_base,
                                                                      const uint16_t* __restrict__ slice_units, int64_t* __restrict__ unit_off,
                                                                      unsigned long long* __restrict__ first_bad, unsigned long long* __restrict__ order_bad) {
    const int64_t n_tiles = (n + kUtf8Tile - 1) / kUtf8Tile;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * kUtf8Threads + threadIdx.x; i < n_off; i += static_cast<int64_t>(gridDim.x) * kUtf8Threads) {
        const int64_t o = byte_off[i], b = o - base;
        if (order_bad && i + 1 < n_off && byte_off[i + 1] < o) atomicMin(order_bad, static_cast<unsigned long long>(i));
        int64_t u;
        if (b <= 0 || b > n) {  // the piece start (an empty piece too: nothing was scanned), or not an offset of the piece
            u = 0;
        } else if (b == n) {
            u = tile_base[n_tiles];
        } else {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(src + (b & ~int64_t(15))));
            const uint32_t x[4] = {v.x, v.y, v.z, v.w};
            uint32_t lead = 0, four = 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                lead |= (byte_bits(__vcmpeq4(x[q] & 0xC0C0C0C0u, 0x80808080u)) ^ 0xFu) << (4 * q);
                four |= byte_bits(__vcmpgeu4(x[q], 0xF0F0F0F0u)) << (4 * q);
            }
            const uint32_t k = static_cast<uint32_t>(b & 15), before = (1u << k) - 1u;
            u = tile_base[b / kUtf8Tile] + slice_units[b / kUtf8PerThread] + __popc(lead & before) + __popc(four & lead & before);
            if (!((lead >> k) & 1u)) {  // b cuts a sequence, or starts with a stray continuation byte
                int64_t bad = b;
                for (int back = 1; back <= 3 && b - back >= 0; ++back) {
                    const uint32_t pb = __ldg(src + b - back);
                    if ((pb & 0xC0u) != 0x80u) {
                        const int len = pb >= 0xF0u ? 4 : pb >= 0xE0u ? 3 : pb >= 0xC0u ? 2 : 1;
                        if (len > back) bad = b - back;
                        break;
                    }
                }
                atomicMin(first_bad, static_cast<unsigned long long>(bad));
            }
        }
        unit_off[i] = u;
    }
}

__global__ void __launch_bounds__(kUtf8Threads) utf8_write_kernel(const uint8_t* __restrict__ src, int64_t n, const int64_t* __restrict__ tile_base,
                                                                 uint16_t* __restrict__ dst) {
    __shared__ uint32_t s_warp[kUtf8Threads / 32];
    const int64_t n_tiles = (n + kUtf8Tile - 1) / kUtf8Tile;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t p0 = tile * kUtf8Tile + static_cast<int64_t>(threadIdx.x) * kUtf8PerThread;
        __align__(16) uint8_t b[kUtf8PerThread];
        uint32_t units = 0;
        if (p0 < n) {
            if (p0 + kUtf8PerThread <= n) {
                *reinterpret_cast<uint4*>(b) = __ldg(reinterpret_cast<const uint4*>(src + p0));
            } else {
                for (int k = 0; k < kUtf8PerThread; ++k) b[k] = p0 + k < n ? __ldg(src + p0 + k) : 0x80;
            }
            for (int k = 0; k < kUtf8PerThread; ++k) units += (b[k] & 0xC0u) == 0x80u ? 0u : (b[k] >= 0xF0u ? 2u : 1u);
        }
        // exclusive prefix of `units` over the threads of the tile
        uint32_t incl = units;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= static_cast<uint32_t>(o)) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint32_t before = 0;
        for (uint32_t w = 0; w < warp; ++w) before += s_warp[w];
        __syncthreads();
        if (p0 < n) {
            int64_t at = tile_base[tile] + before + incl - units;
            for (int k = 0; k < kUtf8PerThread; ++k) {
                const uint32_t c = b[k];
                if ((c & 0xC0u) == 0x80u) continue;
                const int64_t p = p0 + k;
                if (p >= n) break;
                auto next = [&](int j) -> uint32_t {  // continuation byte j of the sequence (validated by pass 1)
                    return (k + j < kUtf8PerThread ? b[k + j] : byte_at(src, p + j, n)) & 0x3Fu;
                };
                if (c < 0x80u) {
                    dst[at++] = static_cast<uint16_t>(c);
                } else if (c < 0xE0u) {
                    dst[at++] = static_cast<uint16_t>(((c & 0x1Fu) << 6) | next(1));
                } else if (c < 0xF0u) {
                    dst[at++] = static_cast<uint16_t>(((c & 0x0Fu) << 12) | (next(1) << 6) | next(2));
                } else {
                    const uint32_t cp = (((c & 0x07u) << 18) | (next(1) << 12) | (next(2) << 6) | next(3)) - 0x10000u;
                    dst[at++] = static_cast<uint16_t>(0xD800u + (cp >> 10));
                    dst[at++] = static_cast<uint16_t>(0xDC00u + (cp & 0x3FFu));
                }
            }
        }
    }
}

// ------------------------------------------------------------------ byte coordinates (gorp_extract_text_utf8_bytes)

// K1's count pass over BYTES: 32 bytes per thread (two 128-bit loads), '\n' found four bytes at a time (__vcmpeq4), one
// 32-bit mask word per thread — the layout of nl_count_mask_kernel, so its scatter pass (nl_scatter_mask_kernel) turns the
// masks into byte line offsets unchanged.
__global__ void __launch_bounds__(kUtf8Threads) utf8_nl_count_mask_kernel(const uint8_t* __restrict__ src, int64_t n,
                                                                         uint32_t* __restrict__ tile_counts, uint32_t* __restrict__ masks) {
    static_assert(kNlTile == kUtf8Threads * 32, "one mask word = 32 bytes");
    const int64_t mine = static_cast<int64_t>(blockIdx.x) * kNlTile + static_cast<int64_t>(threadIdx.x) * 32;
    uint32_t mask = 0;  // bit k: byte mine+k is '\n'
    if (mine + 32 <= n) {
        const uint4* p = reinterpret_cast<const uint4*>(src + mine);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) mask |= byte_bits(__vcmpeq4(w[j], 0x0A0A0A0Au)) << (4 * j);
    } else {
        for (int k = 0; k < 32; ++k)
            if (mine + k < n && src[mine + k] == 0x0A) mask |= 1u << k;
    }
    masks[static_cast<int64_t>(blockIdx.x) * kUtf8Threads + threadIdx.x] = mask;
    __shared__ uint32_t s_warp[kUtf8Threads / 32];
    const uint32_t total = block_sum(static_cast<uint32_t>(__popc(mask)), s_warp);
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

// Result rows of one piece in byte coordinates: ONE WARP per group of 32 lines.
//  - lane l takes line 32 g + l: writes its byte offset (+ bias); the line is ASCII exactly when its byte length equals its
//    unit length (a 2- or 3-byte sequence is 1 unit, a 4-byte sequence 2), and then its row is valid as it is: the warp
//    copies the rows of the group's ASCII lines (coalesced).
//  - every other line of the group is converted by the whole warp: the row's boundaries (unit offsets) are sorted in
//    shared memory (bitonic, <= 64 keys), then the warp walks the line in 1024-byte windows, lane l counting the units of
//    32 bytes; a warp scan gives the unit offset at each lane's slice, and the lane places the sorted boundaries that fall
//    in its slice at the sequence starts that carry them. The walk stops once the last boundary is placed.
//    Work per line: O(len / 32) per lane + the sort; a 100 KB line is 100 window steps of the warp, not a serial walk.
// A boundary never falls inside a surrogate pair of text decoded from well-formed UTF-8 (no lone surrogates; capture
// automata consume whole pairs), so every boundary lands on a sequence start.
// kLines (gorp_extract_lines_utf8): no separator; byte_off is the caller's offsets [n_lines + 1] (the piece starts at byte
// `bias` of the caller's buffer), and out_off is a copy of them, or nullptr when the caller returns its own offsets.
constexpr int kRowsThreads = 256;

template <bool kLines>
__global__ void __launch_bounds__(kRowsThreads) utf8_rows_kernel(Utf8RowsParams P) {
    __shared__ unsigned long long s_keys[kRowsThreads / 32][64];
    const uint32_t lane = threadIdx.x & 31u;
    unsigned long long* keys = s_keys[threadIdx.x >> 5];
    const uint32_t stride = P.stride;
    const int64_t n = P.n_lines;
    const bool write_off = !kLines || P.out_off;
    if (n == 0 && write_off && blockIdx.x == 0 && threadIdx.x == 0) P.out_off[0] = kLines ? P.byte_off[0] : P.bias + P.end_off;
    const int64_t n_groups = (n + 31) / 32;
    const int64_t warps = static_cast<int64_t>(gridDim.x) * (kRowsThreads / 32);
    for (int64_t g = static_cast<int64_t>(blockIdx.x) * (kRowsThreads / 32) + (threadIdx.x >> 5); g < n_groups; g += warps) {
        const int64_t line = g * 32 + lane;
        const bool valid = line < n;
        int64_t u0 = 0, u1 = 0, b0 = 0, b1 = 0;
        if (valid) {
            u0 = P.unit_off[line];
            u1 = P.unit_off[line + 1];
            if constexpr (kLines) {
                b0 = P.byte_off[line] - P.bias;
                b1 = P.byte_off[line + 1] - P.bias;
            } else {
                b0 = line == 0 ? 0 : P.byte_off[line];
                b1 = line + 1 == n ? P.end_off : P.byte_off[line + 1];
            }
            if (write_off) {
                P.out_off[line] = b0 + P.bias;
                if (line + 1 == n) P.out_off[n] = b1 + P.bias;
            }
        }
        if (stride == 0) continue;
        uint32_t other = __ballot_sync(0xffffffffu, valid && b1 - b0 != u1 - u0);
        {   // rows of the ASCII lines: as they are
            const int64_t r0 = g * 32, cnt = (n - r0 < 32 ? n - r0 : 32) * stride;
            const int32_t* __restrict__ in = P.spans + r0 * stride;
            int32_t* __restrict__ out = P.out_spans + r0 * stride;
            for (uint32_t i = lane; i < cnt; i += 32)
                if (!((other >> (i / stride)) & 1u)) out[i] = in[i];
        }
        while (other) {
            const int j = __ffs(other) - 1;
            other &= other - 1;
            const int64_t ln = g * 32 + j;
            const int64_t lu0 = __shfl_sync(0xffffffffu, u0, j), lu1 = __shfl_sync(0xffffffffu, u1, j);
            const int64_t lb0 = __shfl_sync(0xffffffffu, b0, j), lb1 = __shfl_sync(0xffffffffu, b1, j);
            constexpr int64_t sep = kLines ? 0 : 1;
            const int64_t len_u = lu1 - lu0 - sep, len_b = lb1 - lb0 - sep;
            const int32_t* __restrict__ in = P.spans + ln * stride;
            int32_t* __restrict__ out = P.out_spans + ln * stride;
            // keys (unit offset << 8 | slot) of the boundaries inside the line; -1 stays -1, the line's end maps to its byte length
            uint32_t m = 0;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const uint32_t s = lane + 32u * r;
                const int32_t v = s < stride ? in[s] : -1;
                const bool key = v >= 0 && v < len_u;
                keys[s] = key ? (static_cast<unsigned long long>(v) << 8) | s : ~0ull;
                if (s < stride && !key) out[s] = v < 0 ? -1 : static_cast<int32_t>(len_b);
                m += __popc(__ballot_sync(0xffffffffu, key));
            }
            __syncwarp();
            for (uint32_t k = 2; k <= 64; k <<= 1)  // bitonic sort of the 64 keys (padding ~0 sorts last)
                for (uint32_t h = k >> 1; h > 0; h >>= 1) {
                    const uint32_t i = (lane / h) * 2 * h + (lane % h), p = i + h;
                    const unsigned long long x = keys[i], y = keys[p];
                    if (((i & k) == 0) == (x > y)) {
                        keys[i] = y;
                        keys[p] = x;
                    }
                    __syncwarp();
                }
            if (m == 0) continue;
            const int64_t last = static_cast<int64_t>(keys[m - 1] >> 8);
            int64_t base = 0;  // units of the line before the current window
            for (int64_t w = lb0 & ~int64_t(31); w < lb0 + len_b && base <= last; w += 1024) {
                const int64_t s0 = w + 32 * static_cast<int64_t>(lane);
                uint32_t lead = 0, four = 0;
                if (s0 < lb0 + len_b && s0 + 32 > lb0) {
                    // (the second half only when the line reaches into it: the bytes end where the caller's buffer may end)
                    const uint4* p = reinterpret_cast<const uint4*>(P.bytes + s0);
                    const uint4 a = __ldg(p), b = s0 + 16 < lb0 + len_b ? __ldg(p + 1) : make_uint4(0, 0, 0, 0);
                    const uint32_t x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        lead |= (byte_bits(__vcmpeq4(x[q] & 0xC0C0C0C0u, 0x80808080u)) ^ 0xFu) << (4 * q);
                        four |= byte_bits(__vcmpgeu4(x[q], 0xF0F0F0F0u)) << (4 * q);
                    }
                    // only the bytes of the line
                    const int64_t lo = lb0 - s0, hi = lb0 + len_b - s0;
                    const uint32_t keep = (lo > 0 ? ~0u << lo : ~0u) & (hi < 32 ? (1u << hi) - 1u : ~0u);
                    lead &= keep;
                    four &= lead;
                }
                const uint32_t units = __popc(lead) + __popc(four);
                uint32_t incl = units;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= static_cast<uint32_t>(o)) incl += t;
                }
                int64_t c = base + (incl - units);  // unit offset of the first sequence that starts in this lane's slice
                const int64_t c_end = c + units;
                // first key >= c (binary search over the m sorted keys)
                uint32_t lo = 0, hi = m;
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (static_cast<int64_t>(keys[mid] >> 8) < c) lo = mid + 1;
                    else hi = mid;
                }
                if (lo < m && static_cast<int64_t>(keys[lo] >> 8) < c_end) {
                    uint32_t bits = lead;
                    while (bits && lo < m) {
                        const int k = __ffs(bits) - 1;
                        bits &= bits - 1;
                        unsigned long long key;
                        while (lo < m && static_cast<int64_t>((key = keys[lo]) >> 8) <= c) {
                            out[key & 0xFFu] = static_cast<int32_t>(s0 + k - lb0);
                            ++lo;
                        }
                        c += 1 + ((four >> k) & 1u);
                    }
                }
                base += __shfl_sync(0xffffffffu, incl, 31);
            }
            __syncwarp();
        }
    }
}

}  // namespace

int64_t utf8_tiles(int64_t n_bytes) { return (n_bytes + kUtf8Tile - 1) / kUtf8Tile; }

void k_utf8_count_newlines_masks(const Launch& L, const uint8_t* src, int64_t n, uint32_t* tile_counts, uint32_t* masks) {
    if (n <= 0) return;
    utf8_nl_count_mask_kernel<<<static_cast<int>((n + kNlTile - 1) / kNlTile), kUtf8Threads, 0, L.stream>>>(src, n, tile_counts, masks);
}

void k_utf8_rows(const Launch& L, const Utf8RowsParams& P, bool lines) {
    const int64_t want = ((P.n_lines + 31) / 32 + kRowsThreads / 32 - 1) / (kRowsThreads / 32), cap = static_cast<int64_t>(L.sm_count) * 8;
    const int grid = static_cast<int>(want < 1 ? 1 : want < cap ? want : cap);
    if (lines) utf8_rows_kernel<true><<<grid, kRowsThreads, 0, L.stream>>>(P);
    else utf8_rows_kernel<false><<<grid, kRowsThreads, 0, L.stream>>>(P);
}

void k_utf8_count(const Launch& L, const uint8_t* src, int64_t n, uint32_t* tile_counts, unsigned long long* first_bad, uint16_t* slice_units) {
    if (n <= 0) return;
    const int64_t tiles = utf8_tiles(n), cap = static_cast<int64_t>(L.sm_count) * 8;
    const int grid = static_cast<int>(tiles < cap ? tiles : cap);
    if (slice_units) utf8_count_kernel<true><<<grid, kUtf8Threads, 0, L.stream>>>(src, n, tile_counts, first_bad, slice_units);
    else utf8_count_kernel<false><<<grid, kUtf8Threads, 0, L.stream>>>(src, n, tile_counts, first_bad, nullptr);
}

void k_utf8_line_units(const Launch& L, const uint8_t* src, int64_t n, const int64_t* byte_off, int64_t n_off, int64_t base, const int64_t* tile_base,
                       const uint16_t* slice_units, int64_t* unit_off, unsigned long long* first_bad, unsigned long long* order_bad) {
    if (n_off <= 0) return;
    const int64_t want = (n_off + kUtf8Threads - 1) / kUtf8Threads, cap = static_cast<int64_t>(L.sm_count) * 16;
    utf8_line_units_kernel<<<static_cast<int>(want < cap ? want : cap), kUtf8Threads, 0, L.stream>>>(src, n, byte_off, n_off, base, tile_base,
                                                                                                    slice_units, unit_off, first_bad, order_bad);
}

void k_utf8_write(const Launch& L, const uint8_t* src, int64_t n, const int64_t* tile_base, uint16_t* dst) {
    if (n <= 0) return;
    const int64_t tiles = utf8_tiles(n), cap = static_cast<int64_t>(L.sm_count) * 8;
    utf8_write_kernel<<<static_cast<int>(tiles < cap ? tiles : cap), kUtf8Threads, 0, L.stream>>>(src, n, tile_base, dst);
}

}  // namespace gorp
