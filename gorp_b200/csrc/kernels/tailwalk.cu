// K4c — tail walk (sm_100a): the capture half of the text form for extractions that have a tail automaton
// (host/tails.hpp): F_e = minimal DFA of regex_e x capture automaton of e. One walk over the line decides the outcome of
// Gorp.extract for a line whose combined-DFA walk stopped early with candidate e (reference Gorp.java:159-177: MISS when
// regex_e rejects, CAPTURE_FAIL when only java.util.regex rejects, else MATCH) and yields the group spans of
// JDKRegexpCookedExtraction.match/_constructMatch (jdkre/JDKRegexpCookedExtraction.java:36-59).
//
// Work decomposition = kernels/capwalk.cu (lines bucketed by candidate extraction, a CTA takes work items of <= 4096
// lines of ONE extraction, lanes claim lines from the CTA's cursor one line ahead). The extraction's table lives in shared
// memory as directly ASCII-indexed rows of u16 entries,
//
//   per unit :  ent = LDS.U16[row(ent) + 2*unit]          one shared-memory lookup, the only dependent chain
//               STS.U16 slot(ent)[thread] = position + 1    "last position at which command list `slot` fired"
//   per line :  the '\n' column leads to the absorbing row of the line's OUTCOME; a dead transition to the MISS outcome
//
// no class lookup, no trap rows, no register copies. Positions are line-relative and held as u16 (+1, 0 = not written):
// lines of kTailMaxLen units or more are handed to a one-thread-per-line kernel with 32-bit slots (tail_long_kernel).
// A warp works in ROUNDS of `round_iters` walk iterations (16 units each). Everything that is not the walk happens at the
// service point between two rounds, for all lanes that need it at once (so that code runs with many active lanes instead of
// once per lane and iteration): result rows of the lines that ended in the last round (written by the thread that walked
// the line), line starts, claims of the next lines (one record load per line: start, length, id — written by the bucket
// pass). A lane whose line ends inside a round idles until the next service point. The first 32 bytes of a lane's next
// line are loaded into registers and the rest is prefetched into L2 half a round after the claim, so a line start
// never waits for memory.
#include <cstdlib>

#include "device_common.cuh"

namespace gorp {

namespace {

using namespace dev;

__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u16(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(static_cast<unsigned short>(v)) : "memory");
}

// one step on an ASCII unit held in byte kByte (0 or 2) of w. `ra` = byte offset of the current row + rows_abs.
// bytes between the same thread's cells of two consecutive slots. The 32 lanes of a warp cover 16 words of a slot's row (two
// neighbouring lanes share a word): with a stride of 16 words mod 32 the rows of even and odd slots use the two halves of
// the banks, so a lane that stores to another slot than its neighbours (most lanes store to the dummy slot 0) collides at
// most with the lane it shares a word with. The earlier stride (1 word mod 32) put slot s of lane pair k on the bank of
// slot 0 of lane pair k + s: 0.72 extra wavefronts per store (ncu, profiles/README.md round 2).
template <int kT>
struct SlotStride {
    static constexpr uint32_t value = kT * 2 + 64;
    static_assert((value / 4) % 32 == 16, "stride of a slot row: 16 words mod 32");
};

// (A/B, round 2: carrying the last ENTRY instead of the row address, so that the unit's column offset folds into the
// row-address multiply-add — chain LDS -> SHF -> IMAD -> LDS, one IMAD shorter — measured 0.2-0.3 ms SLOWER; not kept.)
template <int kByte, int kT>
__device__ __forceinline__ void tw_step(uint32_t& ra, uint32_t w, uint32_t rows_abs, uint32_t row_bytes, uint32_t slot_abs, uint32_t pos1) {
    uint32_t b, a;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(b) : "r"(w), "n"(kByte == 0 ? 0x4440 : 0x4442));
    asm("mad.lo.u32 %0, %1, 2, %2;" : "=r"(a) : "r"(b), "r"(ra));
    const uint32_t ent = lds_u16(a);
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(ra) : "r"(ent >> 6), "r"(row_bytes), "r"(rows_abs));
    // the store is predicated on a real slot: most units fire no command (slot 0, the dummy), and a warp-wide store in
    // which a few lanes hit other rows than the dummy row cost an extra wavefront (two lanes share a word)
    const uint32_t slot = ent & 63u;
    uint32_t sa;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(sa) : "r"(slot), "n"(SlotStride<kT>::value), "r"(slot_abs));
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p st.shared.u16 [%0], %1; }" ::"r"(sa), "h"(static_cast<unsigned short>(pos1)), "r"(slot) : "memory");
}

// 16 units that hold a unit >= 0x80: unit by unit through the column map (global, L1/L2 resident). A high surrogate
// followed by a low surrogate takes the PAIR column (java.util.regex consumes the pair as one character).
__device__ __noinline__ uint32_t tw_slow16(const TailDev& T, uint32_t ra, const Units16 u, const uint16_t* __restrict__ text, int64_t q,
                                           int64_t n_units, uint32_t rows_abs, uint32_t row_bytes, uint32_t fin_ra, uint32_t slot_abs,
                                           uint32_t pos1, uint32_t kSlotStride) {
    const uint32_t w[8] = {u.a.x, u.a.y, u.a.z, u.a.w, u.b.x, u.b.y, u.b.z, u.b.w};
#pragma unroll 1
    for (int k = 0; k < 16; ++k) {
        if (ra >= fin_ra) break;
        const uint32_t cu = (k & 1) ? (w[k >> 1] >> 16) : (w[k >> 1] & 0xFFFFu);
        uint32_t col = cu;
        if (cu >= 0x80u) {
            col = __ldg(T.xcol + cu);
            if ((cu & 0xFC00u) == 0xD800u) {
                const uint32_t nx = k == 15 ? (q + 16 < n_units ? __ldg(text + q + 16) : 0x0Au)
                                            : ((k & 1) ? (w[(k + 1) >> 1] & 0xFFFFu) : (w[k >> 1] >> 16));
                if ((nx & 0xFC00u) == 0xDC00u) col = __ldg(T.pair_col + col);
            }
        }
        const uint32_t ent = lds_u16(ra + col * 2);
        ra = (ent >> 6) * row_bytes + rows_abs;
        sts_u16(slot_abs + (ent & 63u) * kSlotStride, pos1 + k);
    }
    return ra;
}

// Lines form (List<String>): 16 units with explicit line bounds — the line ends at `end` (the terminator column is applied
// there instead of reading a unit), a '\n' before `end` is line content (its own column), a surrogate pair must lie inside
// the line.
__device__ __noinline__ uint32_t tw_bounded16(const TailDev& T, uint32_t ra, const Units16 u, const uint16_t* __restrict__ text, int64_t q,
                                              int64_t end, uint32_t rows_abs, uint32_t row_bytes, uint32_t fin_ra, uint32_t slot_abs,
                                              uint32_t pos1, uint32_t kSlotStride) {
    const uint32_t w[8] = {u.a.x, u.a.y, u.a.z, u.a.w, u.b.x, u.b.y, u.b.z, u.b.w};
#pragma unroll 1
    for (int k = 0; k < 16; ++k) {
        if (ra >= fin_ra) break;
        const int64_t p = q + k;
        uint32_t col = 0x0Au;  // at the end of the line: the terminator column
        if (p < end) {
            const uint32_t cu = (k & 1) ? (w[k >> 1] >> 16) : (w[k >> 1] & 0xFFFFu);
            col = cu;
            if (cu == 0x0Au) {
                col = T.nl_data_col;
            } else if (cu >= 0x80u) {
                col = __ldg(T.xcol + cu);
                if ((cu & 0xFC00u) == 0xD800u && p + 1 < end) {
                    const uint32_t nx = k == 15 ? __ldg(text + q + 16) : ((k & 1) ? (w[(k + 1) >> 1] & 0xFFFFu) : (w[k >> 1] >> 16));
                    if ((nx & 0xFC00u) == 0xDC00u) col = __ldg(T.pair_col + col);
                }
            }
        }
        const uint32_t ent = lds_u16(ra + col * 2);
        ra = (ent >> 6) * row_bytes + rows_abs;
        sts_u16(slot_abs + (ent & 63u) * kSlotStride, pos1 + k);
    }
    return ra;
}

constexpr uint32_t kTwBins = 1024;    // bins of the per-item sort: (group of records, 32 length classes)
constexpr uint32_t kTwMaxMulti = 64;  // group boundaries with several writers, per extraction (else the table is refused)

// kAll: the fused walk — one table for every line, consecutive lines straight from the line index (no buckets, no records)
template <bool kLines, int kT, bool kAll>
__global__ void __launch_bounds__(kT, 2) tailwalk_kernel(TailWalkParams P) {
    constexpr uint32_t kSlotStride = SlotStride<kT>::value;
    constexpr int kTailWalkThreads = kT;
    // [table][recipes][outcome codes][kAll: lines per outcome][several-writer list][init list][slots: (max_slots + 2) x kSlotStride]
    extern __shared__ __align__(16) unsigned char s_mem[];
    __shared__ uint32_t s_item, s_cursor, s_loaded, s_n_multi;
    const TailDev& T = P.t;
    const uint32_t stride = T.span_stride;
    const uint32_t tab_bytes = T.max_table_bytes;
    uint32_t* s_res = reinterpret_cast<uint32_t*>(s_mem + tab_bytes);
    int32_t* s_oext = reinterpret_cast<int32_t*>(s_res + T.max_res);
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(s_oext + T.max_outcomes);  // kAll: lines per outcome of the one table
    uint32_t* s_multi = s_hist + (kAll ? T.max_outcomes : 0u);  // (outcome << 16 | k), packed writers
    uint8_t* s_init = reinterpret_cast<uint8_t*>(s_multi + 2 * kTwMaxMulti);
    unsigned char* s_slots = reinterpret_cast<unsigned char*>(s_init + 64);
    // [order: kCapItemLines x u16][length bins: kTwBins x u32] — the item's lines sorted by length (see below)
    uint16_t* s_order = reinterpret_cast<uint16_t*>(s_slots + (((T.max_slots + 2) * kSlotStride + 15u) & ~15u));
    uint32_t* s_bins = reinterpret_cast<uint32_t*>(s_order + kCapItemLines);
    const uint32_t rows_abs = static_cast<uint32_t>(__cvta_generic_to_shared(s_mem));
    const uint32_t slot_abs = static_cast<uint32_t>(__cvta_generic_to_shared(s_slots)) + threadIdx.x * 2;
    // slots 0..max_slots-1 of the table (0 = dummy), then ZERO (never written: reads as "no writer") and LEN
    const uint32_t zero_off = T.max_slots * kSlotStride, len_off = zero_off + kSlotStride;
    const uint32_t row_bytes = T.row_bytes;
    const uint32_t lane = threadIdx.x & 31u, lt_mask = (1u << lane) - 1u;
    const uint32_t n_all = kAll ? static_cast<uint32_t>(P.n_lines) : 0u;
    const uint32_t item_lines = kAll ? P.item_lines : kCapItemLines;
    const uint32_t n_items = kAll ? (n_all + item_lines - 1) / item_lines : *P.n_items;
    if (kAll)
        for (uint32_t i = threadIdx.x; i < T.max_outcomes; i += kT) s_hist[i] = 0;
    const uint32_t round_iters = P.round_iters;
    const bool pf_ahead = !(P.flags & 8u);
    if (threadIdx.x == 0) s_loaded = 0xFFFFFFFFu;
    sts_u16(slot_abs + zero_off, 0u);

    // copies the table of an extraction (and its recipes / outcome codes / init list) to shared memory — called by the whole CTA
    auto load_table = [&](const TailExt& x) {
        const uint32_t n16 = ((x.fin_base + x.n_outcomes) * row_bytes + 15u) / 16u;
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(T.image) + x.tab_off);
        uint4* dst = reinterpret_cast<uint4*>(s_mem);
        for (uint32_t i = threadIdx.x; i < n16; i += kTailWalkThreads) dst[i] = __ldg(src + i);
        if (threadIdx.x == 0) s_n_multi = 0;
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < x.n_outcomes; i += kTailWalkThreads) s_oext[i] = __ldg(T.oext + x.oext_off + i);
        for (uint32_t i = threadIdx.x; i < x.n_outcomes * stride; i += kTailWalkThreads) {
            const uint32_t rec = __ldg(T.res + x.res_off + i);
            const bool match = __ldg(T.oext + x.oext_off + i / stride) >= 0;
            // a recipe becomes the byte offset of the slot that holds the boundary + 1:
            // no writer / not a MATCH outcome -> ZERO, the line length -> LEN, one writer -> its slot,
            // several writers -> ZERO here and an entry in the several-writer list
            uint32_t off = zero_off;
            if (match && rec == 0xFFu) {
                off = len_off;
            } else if (match && rec && rec < 256u) {
                off = rec * kSlotStride;
            } else if (match && rec) {
                const uint32_t at = atomicAdd(&s_n_multi, 1u);
                if (at < kTwMaxMulti) {
                    s_multi[2 * at] = ((i / stride) << 16) | (i % stride);
                    s_multi[2 * at + 1] = rec;
                }
            }
            s_res[i] = off;
        }
        for (uint32_t i = threadIdx.x; i < x.n_init; i += kTailWalkThreads) s_init[i] = __ldg(T.init_slots + x.init_off + i);
    };
    // "all" mode: one table for the whole launch — loaded once, and every WARP takes work items on its own (no barrier between
    // items, no shared cursor: the lanes that run out of lines at the end of an item idle for half a line out of item_lines / 32)
    if (kAll) {
        load_table(T.ext[0]);
        __syncthreads();
    }
    for (;;) {
        uint32_t item = 0;
        if (kAll) {
            if (lane == 0) item = atomicAdd(P.item_ticket, 1u);
            item = __shfl_sync(0xffffffffu, item, 0);
        } else {
            __syncthreads();  // the previous item is finished (its table and s_item / s_cursor are free)
            if (threadIdx.x == 0) s_item = atomicAdd(P.item_ticket, 1u);
            __syncthreads();
            item = s_item;
        }
        if (item >= n_items) break;
        CapItem it;
        if (kAll) {
            it.ext = 0;
            it.begin = item * item_lines;
            it.end = min(it.begin + item_lines, n_all);
        } else {
            it = P.items[item];
        }
        const TailExt x = T.ext[it.ext];
        if (!x.available) continue;  // the bucketed capture walk (kernels/capwalk.cu) takes the items of this extraction
        if (!kAll && s_loaded != it.ext) load_table(x);
        // The lanes of a warp walk in lock-step, so a warp is as slow as its longest line. Optional (P.flags & 16, off by default:
        // see profiles/README.md round 2 — the walk is bound by shared-memory wavefronts, not by idle lanes): the item's lines
        // are handed out sorted by DECREASING length inside groups of 2^G consecutive records (counting sort by the number of
        // 16-unit blocks a line touches, in shared memory), so that the 32 lines a warp claims together end within the same
        // iteration or two while staying close to each other in the text. The second pass finds the records in L2.
        const uint32_t n_it = it.end - it.begin;
        const bool sorted = !kAll && (P.flags & 16u) != 0;
        if (sorted) {
            const uint32_t G = max(7u, min(12u, (P.flags >> 8) & 15u ? (P.flags >> 8) & 15u : 8u));
            for (uint32_t i = threadIdx.x; i < kTwBins; i += kTailWalkThreads) s_bins[i] = 0;
            __syncthreads();
            const uint4* recs4 = reinterpret_cast<const uint4*>(P.recs) + it.begin;
            auto key_of = [&](uint32_t i) {  // (group of records, 31 - 16-unit blocks the line touches)
                uint32_t lo, len;
                if (kAll) {
                    const int64_t a0 = __ldg(P.line_off + it.begin + i), a1 = __ldg(P.line_off + it.begin + i + 1);
                    lo = static_cast<uint32_t>(a0) & 15u;
                    len = static_cast<uint32_t>(min(a1 - a0, int64_t(0xFFFF)));
                } else {
                    const uint4 r = __ldg(recs4 + i);
                    lo = r.x & 15u;
                    len = min(r.w, 0xFFFFu);
                }
                return ((i >> G) << 5) + 31u - min((lo + len) >> 4, 31u);
            };
            for (uint32_t i = threadIdx.x; i < n_it; i += kTailWalkThreads) atomicAdd(&s_bins[key_of(i)], 1u);
            __syncthreads();
            if (threadIdx.x < 32) {  // exclusive scan of the kTwBins counts: lane l owns bins [32 l, 32 l + 32)
                uint32_t sum = 0;
                for (uint32_t k = 0; k < kTwBins / 32; ++k) sum += s_bins[lane * (kTwBins / 32) + k];
                uint32_t incl = sum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= static_cast<uint32_t>(o)) incl += t;
                }
                uint32_t run = incl - sum;
                for (uint32_t k = 0; k < kTwBins / 32; ++k) {
                    const uint32_t c = s_bins[lane * (kTwBins / 32) + k];
                    s_bins[lane * (kTwBins / 32) + k] = run;
                    run += c;
                }
            }
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < n_it; i += kTailWalkThreads)
                s_order[atomicAdd(&s_bins[key_of(i)], 1u)] = static_cast<uint16_t>(i);
        }
        uint32_t wcursor = it.begin;  // kAll: the warp's own cursor (warp-uniform)
        if (!kAll) {
            if (threadIdx.x == 0) s_cursor = it.begin;
            __syncthreads();
            if (threadIdx.x == 0) s_loaded = it.ext;
        }

        const int32_t cand = static_cast<int32_t>(it.ext);
        const uint32_t fin_ra = x.fin_base * row_bytes + rows_abs;
        const uint32_t inv_row_bytes = 0xFFFFFFFFu / row_bytes + 1u;
        const uint32_t skip_ra = x.n_states * row_bytes + rows_abs;  // SKIP_1; SKIP_k = skip_ra + (k - 1) * row_bytes
        const uint32_t n_multi = min(s_n_multi, kTwMaxMulti);

        // writes the result row of a finished line (the thread's own; rows are `stride` int32): every entry is
        // "what its slot holds" - 1 (ZERO slot: -1), the several-writer boundaries are patched afterwards
        auto flush = [&](uint32_t fline, uint32_t outcome) {
            const int32_t code = s_oext[outcome];
            if (kAll) {
                P.ext_id[fline] = code;
                atomicAdd(&s_hist[outcome], 1u);
            } else if (code != cand) {  // the candidate did not match after all: MISS (regex_e rejects) or CAPTURE_FAIL
                P.ext_id[fline] = code;
                atomicAdd(P.hist + cand, ~0ull);  // -1
                atomicAdd(P.hist + P.n_ext + (code == -1 ? 0u : 1u), 1ull);
            }
            if (P.flags & 64u) return;  // diagnostics (timing only): no result rows
            int32_t* out = P.spans + static_cast<int64_t>(fline) * stride;
            const uint32_t* res = s_res + outcome * stride;
            auto value = [&](uint32_t off) -> int32_t { return static_cast<int32_t>(lds_u16(slot_abs + off)) - 1; };
            if ((P.flags & 512u) && (stride & 1u) == 0) {  // A/B: 64-bit stores
                for (uint32_t k = 0; k < stride; k += 2) {
                    const uint2 r2 = *reinterpret_cast<const uint2*>(res + k);
                    *reinterpret_cast<int2*>(out + k) = make_int2(value(r2.x), value(r2.y));
                }
            } else if ((stride & 1u) == 0) {
                // rows are 8-byte aligned. A store instruction costs one L1 tag cycle per 32-byte sector and lane (the rows of a
                // warp's lanes are scattered): the row is cut at its sector boundaries — a head piece up to the first boundary,
                // whole sectors (256-bit stores), a tail piece — so every sector is touched once or twice instead of four times
                // (measured: the result rows were 1.5 of the kernel's 7.3 ms on config #4, profiles/README.md round 2)
                const uint32_t g0 = (fline * stride) & 7u;  // position of the row's first entry inside its sector, in entries (even)
                const uint2* res2 = reinterpret_cast<const uint2*>(res);  // recipes two at a time (stride and k are even)
                auto st2 = [&](uint32_t k) {
                    const uint2 r = res2[k >> 1];
                    *reinterpret_cast<int2*>(out + k) = make_int2(value(r.x), value(r.y));
                };
                auto st4 = [&](uint32_t k) {
                    const uint2 r0 = res2[k >> 1], r1 = res2[(k >> 1) + 1];
                    *reinterpret_cast<int4*>(out + k) = make_int4(value(r0.x), value(r0.y), value(r1.x), value(r1.y));
                };
                uint32_t k = 0;
                if ((g0 & 2u) && stride >= 2) st2(0), k = 2;                               // ... to a 16-byte boundary
                if (((g0 + k) & 4u) && stride - k >= 4) st4(k), k += 4;                     // ... to the sector boundary
                for (; k + 8 <= stride; k += 8) {
                    const uint2 r0 = res2[k >> 1], r1 = res2[(k >> 1) + 1], r2 = res2[(k >> 1) + 2], r3 = res2[(k >> 1) + 3];
                    const int32_t v0 = value(r0.x), v1 = value(r0.y), v2 = value(r1.x), v3 = value(r1.y);
                    const int32_t v4 = value(r2.x), v5 = value(r2.y), v6 = value(r3.x), v7 = value(r3.y);
                    if (((g0 + k) & 7u) == 0) {
                        asm volatile("st.global.L2::evict_first.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(out + k), "r"(v0), "r"(v1), "r"(v2),
                                     "r"(v3), "r"(v4), "r"(v5), "r"(v6), "r"(v7)
                                     : "memory");
                    } else {  // a row shorter than the distance to its first sector boundary never got aligned: two 16-byte halves at most
                        int2* o2 = reinterpret_cast<int2*>(out + k);
                        o2[0] = make_int2(v0, v1), o2[1] = make_int2(v2, v3), o2[2] = make_int2(v4, v5), o2[3] = make_int2(v6, v7);
                    }
                }
                if (stride - k >= 4 && ((g0 + k) & 3u) == 0) st4(k), k += 4;
                for (; k < stride; k += 2) st2(k);
            } else {
                for (uint32_t k = 0; k < stride; ++k) out[k] = value(res[k]);
            }
            for (uint32_t i = 0; i < n_multi; ++i) {  // rare: a boundary with several writers = the latest of them
                const uint32_t key = s_multi[2 * i];
                if ((key >> 16) != outcome) continue;
                uint32_t rec = s_multi[2 * i + 1], best = 0;
                for (; rec; rec >>= 8) best = max(best, lds_u16(slot_abs + (rec & 0xFFu) * kSlotStride));
                out[key & 0xFFFFu] = static_cast<int32_t>(best) - 1;
            }
        };

        bool exhausted = false;  // warp-uniform: the item has no unclaimed line left
        bool active = false, has_fin = false;
        uint32_t line = 0, fin_outcome = 0;
        // the lane's line: `a` first unit, `len` units; the walk keeps only a pointer to its current block, the number of
        // blocks that follow it, and the line-relative position (+1) of the block's first unit
        int64_t a = 0;
        uint32_t len = 0, rem = 0, pos1 = 0;
        const uint16_t* tp = P.text;
        bool safe = false;  // every block of the line lies inside the text: plain 256-bit loads
        uint32_t ra = fin_ra;
        Units16 nxt{};  // the block at tp, loaded one iteration ahead
        // the lane's NEXT line: 0 = none, 1 = record requested, 2 = record here, first block requested, rest on its way to L2
        uint32_t nstage = 0;
        uint4 nrec = make_uint4(0, 0, 0, 0);  // LineRec: start (x, y), line id (z), length (w)
        Units16 nfirst{};
        auto load_block = [&](const uint16_t* p, bool inside) -> Units16 {
            if (inside) {
                Units16 r;
                asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                             : "=r"(r.a.x), "=r"(r.a.y), "=r"(r.a.z), "=r"(r.a.w), "=r"(r.b.x), "=r"(r.b.y), "=r"(r.b.z), "=r"(r.b.w)
                             : "l"(p));
                return r;
            }
            return load_units16_l2keep(P.text, p - P.text, P.n_units);  // the last blocks of the text: unit by unit, padded with '\n'
        };
        for (;;) {
            // ================= service point
            if (has_fin) {
                flush(line, fin_outcome);
                has_fin = false;
            }
            if (!active && nstage == 2) {  // start the claimed line
                line = nrec.z;
                a = static_cast<int64_t>(static_cast<uint64_t>(nrec.x) | (static_cast<uint64_t>(nrec.y) << 32));
                len = nrec.w;
                const uint32_t lo = nrec.x & 15u;
                const int64_t q = a - lo;
                tp = P.text + q;
                rem = (lo + len) >> 4;  // blocks after the first, up to the one that holds the line's '\n' (lines form: its end)
                safe = q + 16 * static_cast<int64_t>(rem) + 16 <= P.n_units;
                pos1 = 1u - lo;  // garbage while skipping: only ever stored to the dummy slot
                nxt = nfirst;
                ra = lo ? skip_ra + (lo - 1) * row_bytes : rows_abs;
                for (uint32_t i = 0; i < x.n_init; ++i) sts_u16(slot_abs + s_init[i] * kSlotStride, 0u);
                sts_u16(slot_abs + len_off, len + 1u);
                active = true;
                nstage = 0;
            }
            if (!exhausted) {  // lanes without a next line claim the next entries of the item
                const uint32_t want = __ballot_sync(0xffffffffu, nstage == 0);
                if (want) {
                    uint32_t base = wcursor;
                    if (kAll) {
                        wcursor += static_cast<uint32_t>(__popc(want));
                    } else {
                        if (lane == 0) base = atomicAdd(&s_cursor, static_cast<uint32_t>(__popc(want)));
                        base = __shfl_sync(0xffffffffu, base, 0);
                    }
                    const uint32_t idx = base + static_cast<uint32_t>(__popc(want & lt_mask));
                    if (nstage == 0 && idx < it.end) {
                        const uint32_t at = sorted ? it.begin + s_order[idx - it.begin] : idx;
                        if (kAll) {  // consecutive lines: the record comes straight from the line index
                            const int64_t a0 = __ldg(P.line_off + at), a1 = __ldg(P.line_off + at + 1);
                            const int64_t l = a1 - a0 - (kLines ? 0 : 1);
                            nrec = make_uint4(static_cast<uint32_t>(static_cast<uint64_t>(a0) & 0xFFFFFFFFu), static_cast<uint32_t>(static_cast<uint64_t>(a0) >> 32), at,
                                              static_cast<uint32_t>(l > 0xFFFFFFFFll ? 0xFFFFFFFFll : l));
                        } else {
                            nrec = __ldg(reinterpret_cast<const uint4*>(P.recs) + at);
                        }
                        nstage = 1;
                    }
                    exhausted = base + static_cast<uint32_t>(__popc(want)) >= it.end;
                }
            }
            if (!__any_sync(0xffffffffu, active || nstage != 0)) break;
            // ================= one round of the walk
            for (uint32_t k = 0; k < round_iters; ++k) {
                if (active) {
                    const Units16 u = nxt;
                    if (rem) nxt = load_block(tp + 16, safe);  // in flight during the 16 steps below
                    // ... and the 128-byte line after the next one is asked into L2 just in time: the register load above then
                    // finds its block in L2 (a whole-line prefetch at claim time came too early and was evicted again)
                    if (pf_ahead && (reinterpret_cast<uintptr_t>(tp) & 127u) == 0 && rem >= 4) asm volatile("prefetch.global.L2 [%0];" ::"l"(tp + 64));
                    // lines form: the fast path needs a block that lies inside the line and holds no '\n' (there it is content)
                    const bool plain = !kLines || (rem && (nl_bits4(u.a.x, u.a.y) | nl_bits4(u.a.z, u.a.w) | nl_bits4(u.b.x, u.b.y) | nl_bits4(u.b.z, u.b.w)) == 0u);
                    if (plain && ((u.a.x | u.a.y | u.a.z | u.a.w | u.b.x | u.b.y | u.b.z | u.b.w) & 0xFF80FF80u) == 0u) {
                        tw_step<0, kT>(ra, u.a.x, rows_abs, row_bytes, slot_abs, pos1);
                        tw_step<2, kT>(ra, u.a.x, rows_abs, row_bytes, slot_abs, pos1 + 1);
                        tw_step<0, kT>(ra, u.a.y, rows_abs, row_bytes, slot_abs, pos1 + 2);
                        tw_step<2, kT>(ra, u.a.y, rows_abs, row_bytes, slot_abs, pos1 + 3);
                        tw_step<0, kT>(ra, u.a.z, rows_abs, row_bytes, slot_abs, pos1 + 4);
                        tw_step<2, kT>(ra, u.a.z, rows_abs, row_bytes, slot_abs, pos1 + 5);
                        tw_step<0, kT>(ra, u.a.w, rows_abs, row_bytes, slot_abs, pos1 + 6);
                        tw_step<2, kT>(ra, u.a.w, rows_abs, row_bytes, slot_abs, pos1 + 7);
                        tw_step<0, kT>(ra, u.b.x, rows_abs, row_bytes, slot_abs, pos1 + 8);
                        tw_step<2, kT>(ra, u.b.x, rows_abs, row_bytes, slot_abs, pos1 + 9);
                        tw_step<0, kT>(ra, u.b.y, rows_abs, row_bytes, slot_abs, pos1 + 10);
                        tw_step<2, kT>(ra, u.b.y, rows_abs, row_bytes, slot_abs, pos1 + 11);
                        tw_step<0, kT>(ra, u.b.z, rows_abs, row_bytes, slot_abs, pos1 + 12);
                        tw_step<2, kT>(ra, u.b.z, rows_abs, row_bytes, slot_abs, pos1 + 13);
                        tw_step<0, kT>(ra, u.b.w, rows_abs, row_bytes, slot_abs, pos1 + 14);
                        tw_step<2, kT>(ra, u.b.w, rows_abs, row_bytes, slot_abs, pos1 + 15);
                    } else if (kLines) {
                        ra = tw_bounded16(T, ra, u, P.text, tp - P.text, a + len, rows_abs, row_bytes, fin_ra, slot_abs, pos1, kSlotStride);
                    } else {
                        ra = tw_slow16(T, ra, u, P.text, tp - P.text, P.n_units, rows_abs, row_bytes, fin_ra, slot_abs, pos1, kSlotStride);
                    }
                    tp += 16;
                    pos1 += 16u;
                    --rem;  // (wraps on the last block: the line ends there, `rem` is set again when the next line starts)
                    if (ra >= fin_ra) {  // the line ended inside these 16 units (its '\n', a dead transition, or the end of the text)
                        fin_outcome = __umulhi(ra - fin_ra, inv_row_bytes);  // exact: a small multiple of row_bytes
                        has_fin = true;
                        active = false;
                    }
                }
                if (k == 0 && nstage == 1) {  // the record claimed at the service point is here: get the line's text moving
                    if (nrec.w >= kTailMaxLen) {  // 32-bit positions: tail_long_kernel
                        const uint32_t slot = atomicAdd(P.n_long, 1u);
                        if (slot < P.long_cap) P.long_lines[slot] = nrec.z;
                        nstage = 0;
                    } else {
                        const int64_t na = static_cast<int64_t>(static_cast<uint64_t>(nrec.x) | (static_cast<uint64_t>(nrec.y) << 32));
                        const int64_t p0 = na & ~int64_t(15);
                        nfirst = load_block(P.text + p0, p0 + 16 <= P.n_units);
                        if (pf_ahead && (p0 & ~int64_t(63)) + 64 <= na + nrec.w)  // the 128-byte line after the first block's
                            asm volatile("prefetch.global.L2 [%0];" ::"l"(P.text + (p0 & ~int64_t(63)) + 64));
                        nstage = 2;
                    }
                }
                if (!__any_sync(0xffffffffu, active)) break;
            }
        }
    }
    if (kAll) {  // per-outcome line counts of this CTA -> the histogram bins of their codes
        __syncthreads();
        const TailExt x = T.ext[0];
        for (uint32_t o = threadIdx.x; o < x.n_outcomes; o += kT) {
            const int32_t code = __ldg(T.oext + x.oext_off + o);
            const uint32_t bin = code >= 0 ? static_cast<uint32_t>(code) : (code == -1 ? P.n_ext : P.n_ext + 1u);
            if (s_hist[o]) atomicAdd(P.hist + bin, static_cast<unsigned long long>(s_hist[o]));
        }
    }
}

// Lines of kTailMaxLen units or more: one thread per line, table in global memory, 32-bit slots in local memory.
__global__ void __launch_bounds__(32) tail_long_kernel(TailWalkParams P) {
    const TailDev& T = P.t;
    const uint32_t n = min(*P.n_long, P.long_cap);
    const uint32_t stride = T.span_stride, width = T.width;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t line = P.long_lines[i];
        const int32_t cand = P.all ? 0 : P.ext_id[line];
        if (cand < 0) continue;
        const TailExt x = T.ext[cand];
        const uint16_t* __restrict__ tab = reinterpret_cast<const uint16_t*>(reinterpret_cast<const unsigned char*>(T.image) + x.tab_off);
        uint32_t slots[64];
        for (uint32_t k = 0; k < 64; ++k) slots[k] = 0;
        const int64_t a = P.line_off[line], b = P.line_off[line + 1] - (P.lines_form ? 0 : 1);
        uint32_t row = 0;
        for (int64_t p = a; row < x.fin_base; ++p) {
            const uint32_t cu = p < b && p < P.n_units ? P.text[p] : 0x0Au;  // position b holds the '\n' (or lies beyond the text / the string)
            uint32_t col = cu;
            if (p < b && cu == 0x0Au) {  // lines form only: a '\n' inside the string is content
                col = T.nl_data_col;
            } else if (cu >= 0x80u) {
                col = T.xcol[cu];
                if ((cu & 0xFC00u) == 0xD800u && p + 1 < b && (P.text[p + 1] & 0xFC00u) == 0xDC00u) col = T.pair_col[col];
            }
            const uint32_t ent = tab[static_cast<size_t>(row) * width + col];
            row = ent >> 6;
            slots[ent & 63u] = static_cast<uint32_t>(p - a) + 1u;
        }
        const uint32_t o = row - x.fin_base;
        const int32_t code = T.oext[x.oext_off + o];
        if (P.all) {
            P.ext_id[line] = code;
            atomicAdd(P.hist + (code >= 0 ? static_cast<uint32_t>(code) : (code == -1 ? P.n_ext : P.n_ext + 1u)), 1ull);
        } else if (code != cand) {
            P.ext_id[line] = code;
            atomicAdd(P.hist + cand, ~0ull);
            atomicAdd(P.hist + P.n_ext + (code == -1 ? 0u : 1u), 1ull);
        }
        int32_t* out = P.spans + static_cast<int64_t>(line) * stride;
        for (uint32_t k = 0; k < stride; ++k) {
            uint32_t rec = T.res[x.res_off + o * stride + k];
            int32_t val = -1;
            if (code >= 0 && rec == 0xFFu) {
                val = static_cast<int32_t>(b - a);
            } else if (code >= 0 && rec) {
                uint32_t best = 0;
                for (; rec; rec >>= 8) best = max(best, slots[rec & 0xFFu]);
                val = static_cast<int32_t>(best) - 1;
            }
            out[k] = val;
        }
    }
}

}  // namespace

// the per-item sort (GORP_TAIL_FLAGS & 16) needs its order / bin arrays; without it they take no shared memory
static bool tailwalk_sort_requested() {
    const char* f = std::getenv("GORP_TAIL_FLAGS");
    return f && (std::atoi(f) & 16);
}

size_t tailwalk_smem_bytes(const TailDev& t, int threads) {
    // per outcome: its code and (fused walk) its line count — up to 1008 outcomes: rows are 10-bit ids
    const size_t sort_bytes = tailwalk_sort_requested() ? kCapItemLines * 2 + kTwBins * 4 : 0;
    return static_cast<size_t>(t.max_table_bytes) + static_cast<size_t>(t.max_res) * 4 + static_cast<size_t>(t.max_outcomes) * 8 +
           2 * kTwMaxMulti * 4 + 64 + ((static_cast<size_t>(t.max_slots + 2) * (static_cast<size_t>(threads) * 2 + 64) + 15) & ~size_t(15)) +
           sort_bytes + 16;
}

namespace {

template <bool kLines, int kT, bool kAll>
int tailwalk_warps_per_sm(const TailDev& t) {
    const size_t smem = tailwalk_smem_bytes(t, kT);
    if (smem > 226 * 1024) return 0;
    allow_max_dynamic_smem(tailwalk_kernel<kLines, kT, kAll>);
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tailwalk_kernel<kLines, kT, kAll>, kT, smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return per_sm * kT / 32;
}

template <bool kLines, int kT, bool kAll>
void tailwalk_launch(const Launch& L, const TailWalkParams& P, int per_sm) {
    const size_t smem = tailwalk_smem_bytes(P.t, kT);
    tailwalk_kernel<kLines, kT, kAll><<<L.sm_count * (per_sm < 1 ? 1 : per_sm), kT, smem, L.stream>>>(P);
}

// the CTA size that keeps the most warps resident (the dependent lookup chain of a lane is latency-bound: the more warps,
// the better it is hidden); ties: the smaller CTA. The choice (three occupancy queries and attribute calls) is made once per
// table geometry and host thread: a host-buffer call launches this kernel once per 64 MB piece.
template <bool kLines, bool kAll>
void tailwalk_dispatch(const Launch& L, const TailWalkParams& P) {
    struct Choice {
        size_t key = ~size_t(0);
        int device = -1, forced = -1, threads = 0, per_sm = 0;
    };
    static thread_local Choice ch;
    const size_t key = tailwalk_smem_bytes(P.t, 256);
    int device = 0;
    cudaGetDevice(&device);
    int forced = static_cast<int>(P.prefer_threads);
    if (const char* f = std::getenv("GORP_TAIL_THREADS")) forced = std::atoi(f);
    if (ch.key != key || ch.device != device || ch.forced != forced) {
        const int w256 = tailwalk_warps_per_sm<kLines, 256, kAll>(P.t), w384 = tailwalk_warps_per_sm<kLines, 384, kAll>(P.t),
                  w512 = tailwalk_warps_per_sm<kLines, 512, kAll>(P.t);
        // measured on config #4 (profiles/README.md, round 2): 16 warps 8.5 ms, 24 warps (2 x 384) 7.34 ms, 32 warps (2 x 512) 7.44 ms
        // all mode (consecutive lines, small table): measured on config #2 (profiles/README.md round 2): 3 x 256 threads 10.8 ms,
        // 2 x 384 8.5 ms, 2 x 512 (64 registers) 7.8 ms
        int t = 256;
        if (kAll && forced == 0 && w512 >= 32) t = 512;
        else if (forced == 384 ? w384 > 0 : (forced == 0 && w384 >= 24 && w384 > w256)) t = 384;
        else if (forced == 512 ? w512 > 0 : (forced == 0 && w512 > w384 && w512 > w256)) t = 512;
        else if (forced == 0 && w384 > w256) t = 384;
        ch.key = key;
        ch.device = device;
        ch.forced = forced;
        ch.threads = t;
        ch.per_sm = (t == 512 ? w512 : t == 384 ? w384 : w256) * 32 / t;
    }
    if (ch.threads == 512) tailwalk_launch<kLines, 512, kAll>(L, P, ch.per_sm);
    else if (ch.threads == 384) tailwalk_launch<kLines, 384, kAll>(L, P, ch.per_sm);
    else tailwalk_launch<kLines, 256, kAll>(L, P, ch.per_sm);
}

}  // namespace

void k4c_tailwalk(const Launch& L, const TailWalkParams& P) {
    if (P.all) {
        if (P.lines_form) tailwalk_dispatch<true, true>(L, P);
        else tailwalk_dispatch<false, true>(L, P);
    } else if (P.lines_form) {
        tailwalk_dispatch<true, false>(L, P);
    } else {
        tailwalk_dispatch<false, false>(L, P);
    }
    tail_long_kernel<<<L.sm_count, 32, 0, L.stream>>>(P);
}

}  // namespace gorp
