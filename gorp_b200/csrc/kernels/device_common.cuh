// Device helpers shared by the kernel files (fast.cu, dfawalk.cu, capwalk.cu, tailwalk.cu, ...). Header-only (no -rdc).
#pragma once
#include "kernels.cuh"

namespace gorp {
namespace dev {

__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

__device__ __forceinline__ uint32_t unit_at(const uint4& v, int k) {
    const uint32_t w = (k >> 1) == 0 ? v.x : (k >> 1) == 1 ? v.y : (k >> 1) == 2 ? v.z : v.w;
    return (k & 1) ? (w >> 16) : (w & 0xFFFFu);
}

// ---- text loads, newline masks
// 8 units at text position `pos` (a multiple of 8); units at or beyond n_units read as '\n'
__device__ __forceinline__ uint4 load_chunk(const uint16_t* __restrict__ text, int64_t pos, int64_t n_units) {
    if (pos + 8 <= n_units) return __ldg(reinterpret_cast<const uint4*>(text + pos));
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int64_t p0 = pos + 2 * j, p1 = p0 + 1;
        const uint32_t lo = p0 < n_units ? __ldg(text + p0) : 0x0Au;
        const uint32_t hi = p1 < n_units ? __ldg(text + p1) : 0x0Au;
        w[j] = lo | (hi << 16);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

struct Units16 {
    uint4 a, b;
};
// 16 units at text position `pos` (a multiple of 16); units at or beyond n_units read as '\n'
__device__ __forceinline__ Units16 load_units16(const uint16_t* __restrict__ text, int64_t pos, int64_t n_units) {
    Units16 r;
    if (pos + 16 <= n_units) {
        // the walk is the last use of these 32 bytes: L2 evict-first keeps the not-yet-walked text of the tiles in flight
        asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(r.a.x), "=r"(r.a.y), "=r"(r.a.z), "=r"(r.a.w), "=r"(r.b.x), "=r"(r.b.y), "=r"(r.b.z), "=r"(r.b.w)
                     : "l"(text + pos));
    } else {
        r.a = load_chunk(text, pos, n_units);
        r.b = load_chunk(text, pos + 8, n_units);
    }
    return r;
}

// same, bypassing L1 but with the normal L2 policy
__device__ __forceinline__ Units16 load_units16_l2keep(const uint16_t* __restrict__ text, int64_t pos, int64_t n_units) {
    Units16 r;
    if (pos + 16 <= n_units) {
        asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(r.a.x), "=r"(r.a.y), "=r"(r.a.z), "=r"(r.a.w), "=r"(r.b.x), "=r"(r.b.y), "=r"(r.b.z), "=r"(r.b.w)
                     : "l"(text + pos));
    } else {
        r.a = load_chunk(text, pos, n_units);
        r.b = load_chunk(text, pos + 8, n_units);
    }
    return r;
}

// same as load_units16_l2keep, asking L2 to fetch the whole 128-byte (or 256-byte) neighbourhood: a walker that reads its line
// 32 bytes at a time finds the following blocks in L2, and DRAM serves full bursts instead of one 64-byte atom per 32-byte
// sector request
template <int kPrefetchBytes>
__device__ __forceinline__ Units16 load_units16_l2wide(const uint16_t* __restrict__ text, int64_t pos, int64_t n_units) {
    Units16 r;
    if (pos + 16 <= n_units) {
        if (kPrefetchBytes == 256)
            asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(r.a.x), "=r"(r.a.y), "=r"(r.a.z), "=r"(r.a.w), "=r"(r.b.x), "=r"(r.b.y), "=r"(r.b.z), "=r"(r.b.w)
                         : "l"(text + pos));
        else
            asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(r.a.x), "=r"(r.a.y), "=r"(r.a.z), "=r"(r.a.w), "=r"(r.b.x), "=r"(r.b.y), "=r"(r.b.z), "=r"(r.b.w)
                         : "l"(text + pos));
    } else {
        r.a = load_chunk(text, pos, n_units);
        r.b = load_chunk(text, pos + 8, n_units);
    }
    return r;
}

// same, with the default cache policy: for walkers that come back to the neighbouring sectors of the same 128-byte line
__device__ __forceinline__ Units16 load_units16_keep(const uint16_t* __restrict__ text, int64_t pos, int64_t n_units) {
    Units16 r;
    if (pos + 16 <= n_units) {
        asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(r.a.x), "=r"(r.a.y), "=r"(r.a.z), "=r"(r.a.w), "=r"(r.b.x), "=r"(r.b.y), "=r"(r.b.z), "=r"(r.b.w)
                     : "l"(text + pos));
    } else {
        r.a = load_chunk(text, pos, n_units);
        r.b = load_chunk(text, pos + 8, n_units);
    }
    return r;
}

// bit k (k < 4) = unit k of the pair of words (a, b) is '\n' (0x000A). Low and high bytes are gathered with PRMT, a
// unit is '\n' iff (low ^ 0x0A) | high == 0; exact zero-byte test, then the four flag bits (7, 15, 23, 31) are
// compressed with one multiply.
__device__ __forceinline__ uint32_t nl_bits4(uint32_t a, uint32_t b) {
    const uint32_t lo = __byte_perm(a, b, 0x6420), hi = __byte_perm(a, b, 0x7531);
    const uint32_t t = (lo ^ 0x0A0A0A0Au) | hi;
    const uint32_t z = ~(((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t | 0x7F7F7F7Fu);  // 0x80 in every zero byte of t
    return (((z >> 7) * 0x00204081u) >> 21) & 0xFu;
}

// one combined-DFA step on an ASCII unit held in byte kByte (0 or 2) of w: state = LDS[state + 4*unit]
template <int kByte>
__device__ __forceinline__ uint32_t dfa_step(uint32_t st, uint32_t w) {
    uint32_t b, addr;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(b) : "r"(w), "n"(kByte == 0 ? 0x4440 : 0x4442));
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(addr) : "r"(b), "r"(st));
    return lds32(addr);
}

// one capture-automaton step: class lookup, row lookup, unconditional "register := position" store
// (transitions without a command store into the per-thread dummy register)
template <int kByte>
__device__ __forceinline__ void cap_step(uint32_t& st, uint32_t w, uint32_t cls_abs, uint32_t tab_abs, uint32_t reg_abs,
                                         uint32_t pos) {
    uint32_t b, addr;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(b) : "r"(w), "n"(kByte == 0 ? 0x4440 : 0x4442));
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(addr) : "r"(b), "r"(cls_abs));
    const uint32_t c4 = lds32(addr);
    const uint32_t ent = lds32(tab_abs + st + c4);
    st = ent & 0xFFFCu;
    sts32(reg_abs + (ent >> 16), pos);
}

// DFA, one chunk unit by unit (chunks that hold a unit >= 0x80): class map and plain table in global memory.
// `st` is an absolute shared-memory row address on entry and exit.
static __device__ __noinline__ uint32_t dfa_slow_chunk(const DfaDirectDev& d, uint32_t tbase, uint32_t st, uint4 v) {
    uint32_t row = (st - tbase) >> 9;
#pragma unroll 1
    for (int k = 0; k < 8; ++k) {
        if (row >= d.fin_base) break;
        const uint32_t u = unit_at(v, k);
        if (row >= d.skip_base) {
            row = row == d.skip_base ? 0u : row - 1;
        } else if (u == 0x0Au) {
            row = d.fin_base + 1 + __ldg(d.accept_first + row);
        } else {
            const int32_t t = __ldg(d.trans_plain + row * d.n_classes + __ldg(d.cls + u));
            row = t < 0 ? d.fin_base : static_cast<uint32_t>(t);
        }
    }
    return tbase + (row << 9);
}

// Capture automaton, one chunk unit by unit through the general tables (units >= 0x80, surrogate pairs, transitions
// with several register commands). `q` = text position of the chunk, `a` = text position of the line start; units at
// or beyond n_units read as '\n'. `st` is a fast-tier row offset on entry and exit; the line length is stored to the
// LEN register at the terminating '\n'.
static __device__ __noinline__ uint32_t tdfa_slow_chunk(const CapDev& c, const ExtDev& x, const FastExtDev& fx, uint32_t st,
                                                        const uint16_t* __restrict__ text, int64_t q, int64_t a, int64_t n_units,
                                                        uint32_t reg_abs, uint32_t reg_stride, uint32_t len_off) {
    const uint32_t S = fx.n_states;
    uint32_t row = st / fx.row_bytes;
    const uint32_t n_cols = c.n_classes + 1;
    const uint32_t* __restrict__ tr = c.tdfa_trans + x.trans_off;
    const uint32_t* __restrict__ opo = c.tdfa_op_off + x.opoff_off;
    const uint16_t* __restrict__ ops = c.tdfa_ops + x.ops_off;
#pragma unroll 1
    for (int k = 0; k < 8; ++k) {
        if (row >= S + 7) break;  // DEAD / FRZ
        const int64_t p = q + k;
        const uint32_t u = p < n_units ? __ldg(text + p) : 0x0Au;
        if (row >= S) {  // SKIP_j
            row = row == S ? 0u : row - 1;
            continue;
        }
        const uint32_t pos = static_cast<uint32_t>(p - a);
        if (u == 0x0Au) {
            sts32(reg_abs + len_off, pos);
            row = S + 9 + row;
            break;
        }
        uint32_t sym = __ldg(c.cls + u);
        // a high surrogate followed by a low surrogate is ONE java.util.regex character
        if ((u & 0xFC00u) == 0xD800u && p + 1 < n_units && (__ldg(text + p + 1) & 0xFC00u) == 0xDC00u) sym = c.pair_hi_class;
        const uint32_t ent = __ldg(tr + row * n_cols + sym);
        const uint32_t ol = ent >> 16;
        if (ol) {
            const uint32_t o0 = __ldg(opo + ol), o1 = __ldg(opo + ol + 1);
            for (uint32_t i = o0; i < o1; ++i) {
                const uint32_t op = __ldg(ops + i);
                const uint32_t src = op & 0xFFu;
                const uint32_t val = src == 0xFFu ? pos : lds32(reg_abs + src * reg_stride);
                sts32(reg_abs + (op >> 8) * reg_stride, val);
            }
        }
        row = ent & 0xFFFFu;
        if (row == S) row = S + 7;  // the general table's dead row index is S
    }
    return row * fx.row_bytes;
}

}  // namespace dev
}  // namespace gorp
