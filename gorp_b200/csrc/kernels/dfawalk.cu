// K2b — line-walk DFA kernel (sm_100a): the combined-DFA scan over an existing line index (K1's, or the caller's offsets
// in the List<String> form). Stands in for PolyMatcher.match + Automata.step/accept (reference autom/PolyMatcher.java:123-133,
// autom/Automata.java:133-139) and the first-index dispatch of Gorp.java:166-167; the capture half runs afterwards, bucketed
// by extraction (kernels/capwalk.cu, kernels/tailwalk.cu).
//
// The automaton is the class-indexed combined DFA (u16 next-row entries, K = classes + 1 columns, the last column is '\n'),
// or its early-exit variant when the tail walk follows (host/walktables.hpp); it lives in shared memory when it fits,
// otherwise it is read through L1/L2 (template kSmem):
//     rows [0,S) states | S = DEADSCAN (dead, keeps scanning to the line's '\n') | S+1..S+15 = SKIP_1..15 (units that
//     precede the line in its first 32-byte block) | fin_base = S+16: FIN(-1), FIN(0..E-1) absorbing outcome rows
// A WARP takes work items of kLineItemLines consecutive lines, every lane walks one line at a time in 32-byte blocks and
// claims its next line one line ahead (ballot-ranked, no atomics), so lanes stay busy whatever the line lengths are (long or
// ragged lines, 10 KB outliers). A finished line writes its extraction id (or -1; with the early-exit table: the candidate).
#include "device_common.cuh"

namespace gorp {

namespace {

using namespace dev;

__device__ __forceinline__ uint32_t lds16(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// newline mask of 16 units (bit k = unit k is '\n')
__device__ __forceinline__ uint32_t nl_mask16(const Units16& u) {
    return nl_bits4(u.a.x, u.a.y) | (nl_bits4(u.a.z, u.a.w) << 4) | (nl_bits4(u.b.x, u.b.y) << 8) | (nl_bits4(u.b.z, u.b.w) << 12);
}

template <bool kSmem>
__device__ __forceinline__ uint32_t dw_next(uint32_t st, uint32_t cx, uint32_t row_bytes, const unsigned char* __restrict__ tab_g) {
    uint32_t a;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(a) : "r"(st), "r"(row_bytes), "r"(cx));
    if (kSmem) return lds16(a);
    return __ldg(reinterpret_cast<const uint16_t*>(tab_g + a));
}

// one step on an ASCII unit held in byte kByte (0 or 2) of w. s_cx[unit] = byte offset of the unit's column inside a
// row (+ the shared-memory address of the table when kSmem), so the dependent chain is one IMAD + one load.
template <bool kSmem, int kByte>
__device__ __forceinline__ uint32_t dw_step(uint32_t st, uint32_t w, uint32_t cx_abs, uint32_t row_bytes,
                                            const unsigned char* __restrict__ tab_g) {
    uint32_t b, a;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(b) : "r"(w), "n"(kByte == 0 ? 0x4440 : 0x4442));
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(a) : "r"(b), "r"(cx_abs));
    return dw_next<kSmem>(st, lds32(a), row_bytes, tab_g);
}

// the same step through a u16 copy of the column table (256 bytes = 64 words: the 32 lanes of a warp read fewer distinct words
// of fewer rows per bank than with the u32 table: fewer wavefronts per lookup; K2b's walk is bound by them). The entries hold
// the shared-memory address of the unit's column in row 0, which fits 16 bits because the table starts the dynamic area.
template <int kByte>
__device__ __forceinline__ uint32_t dw_step16(uint32_t st, uint32_t w, uint32_t c16_abs, uint32_t row_bytes) {
    uint32_t b, a;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(b) : "r"(w), "n"(kByte == 0 ? 0x4440 : 0x4442));
    asm("mad.lo.u32 %0, %1, 2, %2;" : "=r"(a) : "r"(b), "r"(c16_abs));
    return dw_next<true>(st, lds16(a), row_bytes, nullptr);
}

// 8 units that hold a unit >= 0x80: unit by unit through the full class map (global, L1/L2 resident)
template <bool kSmem>
__device__ __noinline__ uint32_t dw_slow8(const DfaWalkDev& A, uint32_t st, uint4 v, uint32_t cx_abs, uint32_t tab_abs, uint32_t row_bytes,
                                          const unsigned char* __restrict__ tab_g) {
#pragma unroll 1
    for (int k = 0; k < 8; ++k) {
        if (st >= A.fin_base) break;
        const uint32_t u = unit_at(v, k);
        const uint32_t cx = u < 0x80u ? lds32(cx_abs + u * 4) : (kSmem ? tab_abs : 0u) + 2u * __ldg(A.xcls + u);
        st = dw_next<kSmem>(st, cx, row_bytes, tab_g);
    }
    return st;
}

// Lines form (List<String>): 16 units unit by unit with explicit line bounds — a line ends at `end` (no '\n' there: the
// NL column is applied instead of reading a unit) and a '\n' before `end` is line content (its class through the full map).
template <bool kSmem>
__device__ __noinline__ uint32_t dw_bounded16(const DfaWalkDev& A, uint32_t st, const Units16 u, int64_t q, int64_t a, int64_t end,
                                              uint32_t cx_abs, uint32_t tab_abs, uint32_t row_bytes, const unsigned char* __restrict__ tab_g) {
    const uint32_t w[8] = {u.a.x, u.a.y, u.a.z, u.a.w, u.b.x, u.b.y, u.b.z, u.b.w};
#pragma unroll 1
    for (int k = 0; k < 16; ++k) {
        if (st >= A.fin_base) break;
        const int64_t p = q + k;
        uint32_t cx;
        if (p >= end) {
            cx = lds32(cx_abs + 0x0Au * 4);  // the NL column: what a '\n'-terminated line reads at its end
        } else {
            const uint32_t cu = (k & 1) ? (w[k >> 1] >> 16) : (w[k >> 1] & 0xFFFFu);
            cx = (cu < 0x80u && cu != 0x0Au) || p < a ? lds32(cx_abs + (cu & 0x7Fu) * 4) : (kSmem ? tab_abs : 0u) + 2u * __ldg(A.xcls + cu);
        }
        st = dw_next<kSmem>(st, cx, row_bytes, tab_g);
    }
    return st;
}

template <bool kSmem, bool kLines>
__global__ void __launch_bounds__(768, 2) linewalk_kernel(LineWalkParams P) {
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t kT = blockDim.x;
    const DfaWalkDev& A = P.a;
    const uint32_t row_bytes = A.K * 2;
    const uint32_t table_bytes = kSmem ? ((A.n_rows * row_bytes + 15u) & ~15u) : 0u;
    uint32_t* s_cx = reinterpret_cast<uint32_t*>(smem + table_bytes);
    uint16_t* s_c16 = reinterpret_cast<uint16_t*>(s_cx + 128);
    const uint32_t tab_abs = static_cast<uint32_t>(__cvta_generic_to_shared(smem));
    const uint32_t cx_abs = static_cast<uint32_t>(__cvta_generic_to_shared(s_cx));
    const uint32_t c16_abs = static_cast<uint32_t>(__cvta_generic_to_shared(s_c16));
    const unsigned char* __restrict__ tab_g = reinterpret_cast<const unsigned char*>(A.table);
    if (kSmem) {
        const uint32_t n16 = (A.n_rows * row_bytes + 15u) / 16u;
        const uint4* src = reinterpret_cast<const uint4*>(A.table);
        uint4* dst = reinterpret_cast<uint4*>(smem);
        for (uint32_t i = threadIdx.x; i < n16; i += kT) dst[i] = __ldg(src + i);
    }
    for (uint32_t i = threadIdx.x; i < 128; i += kT) {
        s_cx[i] = (kSmem ? tab_abs : 0u) + __ldg(A.cls128 + i);
        s_c16[i] = static_cast<uint16_t>(tab_abs + __ldg(A.cls128 + i));
    }
    // the u16 column table serves the fast path when the column addresses of row 0 fit 16 bits (P.flags & 2: A/B, u32 table)
    const bool c16_ok = kSmem && tab_abs + 2u * A.K < 65536u && !(P.flags & 2u);
    __syncthreads();
    const uint32_t fin_base = A.fin_base, skip0 = A.n_states;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int64_t n_items = (P.n_lines + kLineItemLines - 1) / kLineItemLines;

    for (;;) {
        unsigned int item = 0;
        if (lane == 0) item = atomicAdd(P.item_ticket, 1u);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        int64_t cursor = static_cast<int64_t>(item) * kLineItemLines;  // warp-uniform: next unclaimed line of the item
        const int64_t end = cursor + kLineItemLines < P.n_lines ? cursor + kLineItemLines : P.n_lines;
        bool active = false, has_next = false;
        int64_t line = 0, nline = 0, q = 0, na = 0, a = 0, lend = 0, nlend = 0;  // lend: where the line ends (lines form)
        uint32_t st = 0;
        for (;;) {
            if (!active && has_next) {  // start the claimed line
                line = nline;
                a = na;
                lend = nlend;
                q = na & ~int64_t(15);
                const uint32_t lo = static_cast<uint32_t>(na - q);
                st = lo ? skip0 + lo : 0u;
                active = true;
                has_next = false;
            }
            if (cursor < end) {  // lanes without a next line claim the next lines of the item
                const uint32_t want = __ballot_sync(0xffffffffu, !has_next);
                if (want) {
                    const int64_t idx = cursor + __popc(want & lt_mask);
                    if (!has_next && idx < end) {
                        nline = idx;
                        na = __ldg(P.line_off + idx);
                        if (kLines) nlend = __ldg(P.line_off + idx + 1);
                        has_next = true;
                    }
                    cursor += __popc(want);
                }
            }
            if (!__any_sync(0xffffffffu, active || has_next)) break;
            if (active) {
                const Units16 u = P.flags & 1u ? load_units16(P.text, q, P.n_units) : load_units16_l2keep(P.text, q, P.n_units);
                // lines form: the fast path needs a block that lies inside the line and holds no '\n' (there it is content)
                const bool plain = !kLines || (q + 16 <= lend && nl_mask16(u) == 0u);
                const bool ascii = plain && ((u.a.x | u.a.y | u.a.z | u.a.w | u.b.x | u.b.y | u.b.z | u.b.w) & 0xFF80FF80u) == 0u;
                if (ascii && c16_ok) {
                    st = dw_step16<0>(st, u.a.x, c16_abs, row_bytes);
                    st = dw_step16<2>(st, u.a.x, c16_abs, row_bytes);
                    st = dw_step16<0>(st, u.a.y, c16_abs, row_bytes);
                    st = dw_step16<2>(st, u.a.y, c16_abs, row_bytes);
                    st = dw_step16<0>(st, u.a.z, c16_abs, row_bytes);
                    st = dw_step16<2>(st, u.a.z, c16_abs, row_bytes);
                    st = dw_step16<0>(st, u.a.w, c16_abs, row_bytes);
                    st = dw_step16<2>(st, u.a.w, c16_abs, row_bytes);
                    st = dw_step16<0>(st, u.b.x, c16_abs, row_bytes);
                    st = dw_step16<2>(st, u.b.x, c16_abs, row_bytes);
                    st = dw_step16<0>(st, u.b.y, c16_abs, row_bytes);
                    st = dw_step16<2>(st, u.b.y, c16_abs, row_bytes);
                    st = dw_step16<0>(st, u.b.z, c16_abs, row_bytes);
                    st = dw_step16<2>(st, u.b.z, c16_abs, row_bytes);
                    st = dw_step16<0>(st, u.b.w, c16_abs, row_bytes);
                    st = dw_step16<2>(st, u.b.w, c16_abs, row_bytes);
                } else if (ascii) {
                    st = dw_step<kSmem, 0>(st, u.a.x, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 2>(st, u.a.x, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 0>(st, u.a.y, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 2>(st, u.a.y, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 0>(st, u.a.z, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 2>(st, u.a.z, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 0>(st, u.a.w, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 2>(st, u.a.w, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 0>(st, u.b.x, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 2>(st, u.b.x, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 0>(st, u.b.y, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 2>(st, u.b.y, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 0>(st, u.b.z, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 2>(st, u.b.z, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 0>(st, u.b.w, cx_abs, row_bytes, tab_g);
                    st = dw_step<kSmem, 2>(st, u.b.w, cx_abs, row_bytes, tab_g);
                } else if (kLines) {
                    st = dw_bounded16<kSmem>(A, st, u, q, a, lend, cx_abs, tab_abs, row_bytes, tab_g);
                } else {
                    st = dw_slow8<kSmem>(A, st, u.a, cx_abs, tab_abs, row_bytes, tab_g);
                    st = dw_slow8<kSmem>(A, st, u.b, cx_abs, tab_abs, row_bytes, tab_g);
                }
                q += 16;
                if (st >= fin_base) {  // reached the line's '\n' (or the end of the text / of the string)
                    P.ext_id[line] = static_cast<int32_t>(st - fin_base) - 1;
                    active = false;
                }
            }
        }
    }
}

}  // namespace

size_t linewalk_smem_bytes(const DfaWalkDev& a, bool in_smem) {
    return (in_smem ? ((static_cast<size_t>(a.n_rows) * a.K * 2 + 15) & ~size_t(15)) : 0) + 128 * 4 + 128 * 2 + 128;
}

bool k2b_linewalk_plan(const DfaWalkDev& a, uint32_t* threads, bool* in_smem) {
    if (!a.enabled) return false;
    *threads = 768;  // two CTAs per SM (48 warps) when the table leaves room for them
    *in_smem = linewalk_smem_bytes(a, true) <= 200 * 1024;
    return true;
}

template <bool kSmem, bool kLines>
static void launch_linewalk(const Launch& L, const LineWalkParams& P, uint32_t threads, size_t smem) {
    int per_sm = 1;
    allow_max_dynamic_smem(linewalk_kernel<kSmem, kLines>);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, linewalk_kernel<kSmem, kLines>, static_cast<int>(threads), smem);
    linewalk_kernel<kSmem, kLines><<<L.sm_count * (per_sm < 1 ? 1 : per_sm), static_cast<int>(threads), smem, L.stream>>>(P);
}

void k2b_linewalk_scan(const Launch& L, const LineWalkParams& P, uint32_t threads, bool in_smem) {
    const size_t smem = linewalk_smem_bytes(P.a, in_smem);
    if (in_smem) {
        if (P.lines_form) launch_linewalk<true, true>(L, P, threads, smem);
        else launch_linewalk<true, false>(L, P, threads, smem);
    } else {
        if (P.lines_form) launch_linewalk<false, true>(L, P, threads, smem);
        else launch_linewalk<false, false>(L, P, threads, smem);
    }
}

}  // namespace gorp
