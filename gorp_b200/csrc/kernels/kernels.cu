// sm_100a kernels of the gorp batch extraction path. See kernels.cuh for the reference functions they replace.
#include "kernels.cuh"

namespace gorp {
namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
    // streaming 128-bit load: the text is read once per pass, keep it out of L1
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ uint32_t nl_pairs(uint32_t w) {  // 0xFFFF per UTF-16 unit equal to '\n'
    return __vcmpeq2(w, 0x000A000Au);
}

__device__ __forceinline__ uint32_t warp_sum(uint32_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------ K1: newline index
__global__ void __launch_bounds__(kThreads) nl_count_kernel(const uint16_t* __restrict__ text, int64_t n_units,
                                                            uint32_t* __restrict__ tile_counts) {
    const int64_t tile0 = static_cast<int64_t>(blockIdx.x) * kNlTile;
    uint32_t cnt = 0;
    if (tile0 + kNlTile <= n_units) {
        const uint4* src = reinterpret_cast<const uint4*>(text + tile0);
#pragma unroll
        for (int j = 0; j < kNlTile / 8 / kThreads; ++j) {
            uint4 v = ld_stream(src + j * kThreads + threadIdx.x);
            cnt += __popc(nl_pairs(v.x)) + __popc(nl_pairs(v.y)) + __popc(nl_pairs(v.z)) + __popc(nl_pairs(v.w));
        }
        cnt >>= 4;
    } else {
        for (int64_t p = tile0 + threadIdx.x; p < n_units; p += kThreads) cnt += text[p] == 0x0A;
    }
    __shared__ uint32_t warp_tot[kThreads / 32];
    cnt = warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) warp_tot[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) t += warp_tot[w];
        tile_counts[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(kThreads) nl_scatter_kernel(const uint16_t* __restrict__ text, int64_t n_units,
                                                              const int64_t* __restrict__ tile_base,
                                                              int64_t* __restrict__ line_off) {
    constexpr int kPer = kNlTile / kThreads;  // 32 consecutive units per thread
    const int64_t tile0 = static_cast<int64_t>(blockIdx.x) * kNlTile;
    const int64_t mine = tile0 + static_cast<int64_t>(threadIdx.x) * kPer;
    uint32_t mask = 0;  // bit k: unit mine+k is '\n'
    if (mine + kPer <= n_units) {
        const uint4* src = reinterpret_cast<const uint4*>(text + mine);
#pragma unroll
        for (int j = 0; j < kPer / 8; ++j) {
            uint4 v = __ldg(src + j);
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t m = nl_pairs(w[k]);
                mask |= ((m & 1u) | ((m >> 15) & 2u)) << (j * 8 + k * 2);
            }
        }
    } else {
        for (int k = 0; k < kPer; ++k)
            if (mine + k < n_units && text[mine + k] == 0x0A) mask |= 1u << k;
    }
    // block exclusive scan of per-thread counts
    uint32_t cnt = __popc(mask), incl = cnt;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __shared__ uint32_t warp_tot[kThreads / 32];
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    uint32_t base = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w)
        if (w < warp) base += warp_tot[w];
    int64_t slot = 1 + tile_base[blockIdx.x] + base + (incl - cnt);  // line_off[j] = start of line j (j >= 1)
    while (mask) {
        int k = __ffs(mask) - 1;
        mask &= mask - 1;
        line_off[slot++] = mine + k + 1;
    }
}

// K1 with a side product: the count pass also stores the '\n' mask of every 32 units (1 bit per unit), so the scatter
// pass reads 1/16 of the text's bytes instead of the text again (two HBM passes over the text -> one).
__global__ void __launch_bounds__(kThreads) nl_count_mask_kernel(const uint16_t* __restrict__ text, int64_t n_units,
                                                                 uint32_t* __restrict__ tile_counts, uint32_t* __restrict__ masks) {
    constexpr int kPer = kNlTile / kThreads;  // 32 consecutive units per thread
    const int64_t tile0 = static_cast<int64_t>(blockIdx.x) * kNlTile;
    const int64_t mine = tile0 + static_cast<int64_t>(threadIdx.x) * kPer;
    uint32_t mask = 0;  // bit k: unit mine+k is '\n'
    if (mine + kPer <= n_units) {
        const uint4* src = reinterpret_cast<const uint4*>(text + mine);
        uint4 v[kPer / 8];
#pragma unroll
        for (int j = 0; j < kPer / 8; ++j) v[j] = ld_stream(src + j);
#pragma unroll
        for (int j = 0; j < kPer / 8; ++j) {
            const uint32_t w[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t m = nl_pairs(w[k]);
                mask |= ((m & 1u) | ((m >> 15) & 2u)) << (j * 8 + k * 2);
            }
        }
    } else {
        for (int k = 0; k < kPer; ++k)
            if (mine + k < n_units && text[mine + k] == 0x0A) mask |= 1u << k;
    }
    masks[static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x] = mask;
    __shared__ uint32_t warp_tot[kThreads / 32];
    const uint32_t cnt = warp_sum(static_cast<uint32_t>(__popc(mask)));
    if ((threadIdx.x & 31) == 0) warp_tot[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) t += warp_tot[w];
        tile_counts[blockIdx.x] = t;
    }
}

// one WARP per tile (a tile holds ~60 line starts: a block-wide scan with its barrier per tile cost more than the stores):
// lane l takes the 8 mask words of units [256 l, 256 l + 256) of the tile, the warp scans the counts, every lane writes
// the starts of its lines.
__global__ void __launch_bounds__(kThreads) nl_scatter_mask_kernel(const uint32_t* __restrict__ masks, const int64_t* __restrict__ tile_base,
                                                                   int64_t* __restrict__ line_off, int64_t n_tiles) {
    static_assert(kNlTile == 32 * 256, "one lane = 8 mask words");
    const uint32_t lane = threadIdx.x & 31u;
    const int64_t tile = static_cast<int64_t>(blockIdx.x) * (kThreads / 32) + (threadIdx.x >> 5);
    if (tile >= n_tiles) return;
    const uint4* src = reinterpret_cast<const uint4*>(masks + tile * 256) + lane * 2;
    const uint4 a = __ldg(src), b = __ldg(src + 1);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t cnt = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) cnt += __popc(w[j]);
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= static_cast<uint32_t>(o)) incl += t;
    }
    int64_t slot = 1 + tile_base[tile] + (incl - cnt);  // line_off[j] = start of line j (j >= 1)
    const int64_t unit1 = tile * kNlTile + static_cast<int64_t>(lane) * 256 + 1;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        uint32_t m = w[j];
        while (m) {
            const int k = __ffs(m) - 1;
            m &= m - 1;
            line_off[slot++] = unit1 + j * 32 + k;
        }
    }
}

__global__ void nl_finish_kernel(const uint16_t* __restrict__ text, int64_t n_units, const int64_t* __restrict__ total_nl,
                                 int64_t* __restrict__ line_off, int64_t* __restrict__ n_lines_out) {
    const int64_t nl = *total_nl;
    line_off[0] = 0;
    int64_t n_lines = nl;
    if (n_units > 0 && text[n_units - 1] != 0x0A) {  // a final line without '\n' counts
        n_lines = nl + 1;
        line_off[n_lines] = n_units + 1;
    }
    *n_lines_out = n_lines;
}

// ------------------------------------------------------------------ exclusive scan (u32 -> i64)
constexpr int kScanTile = 4096;  // 256 threads x 16

__global__ void __launch_bounds__(kThreads) scan_sums_kernel(const uint32_t* __restrict__ in, int64_t n, int64_t* __restrict__ sums) {
    const int64_t base = static_cast<int64_t>(blockIdx.x) * kScanTile;
    uint32_t s = 0;
    for (int k = threadIdx.x; k < kScanTile; k += kThreads)
        if (base + k < n) s += in[base + k];
    __shared__ uint32_t warp_tot[kThreads / 32];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) warp_tot[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < kThreads / 32; ++w) t += warp_tot[w];
        sums[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024) scan_top_kernel(int64_t* __restrict__ sums, int64_t nb) {
    // single block: exclusive scan of sums[0..nb) in place, sums[nb] = total
    __shared__ int64_t part[1024];
    const int64_t per = (nb + 1023) / 1024;
    const int64_t lo = threadIdx.x * per, hi = min(lo + per, nb);
    int64_t s = 0;
    for (int64_t i = lo; i < hi; ++i) s += sums[i];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t run = 0;
        for (int i = 0; i < 1024; ++i) {
            int64_t t = part[i];
            part[i] = run;
            run += t;
        }
        sums[nb] = run;
    }
    __syncthreads();
    int64_t run = part[threadIdx.x];
    for (int64_t i = lo; i < hi; ++i) {
        int64_t t = sums[i];
        sums[i] = run;
        run += t;
    }
}

__global__ void __launch_bounds__(kThreads) scan_apply_kernel(const uint32_t* __restrict__ in, int64_t n,
                                                              const int64_t* __restrict__ sums, int64_t nb,
                                                              int64_t* __restrict__ out) {
    constexpr int kPer = kScanTile / kThreads;
    const int64_t base = static_cast<int64_t>(blockIdx.x) * kScanTile + static_cast<int64_t>(threadIdx.x) * kPer;
    uint32_t v[kPer];
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        v[k] = (base + k < n) ? in[base + k] : 0u;
        s += v[k];
    }
    uint32_t incl = s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __shared__ uint32_t warp_tot[kThreads / 32];
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    uint32_t wbase = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w)
        if (w < warp) wbase += warp_tot[w];
    int64_t run = sums[blockIdx.x] + wbase + (incl - s);
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        if (base + k < n) out[base + k] = run;
        run += v[k];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = sums[nb];
}

// ------------------------------------------------------------------ line walking shared by K2 / K4
// A line [a, b) is walked in 16-byte aligned chunks of 8 UTF-16 units with ONE loop shape for every thread, so a
// warp never splits into per-thread head/tail code: units of the chunk that lie outside the line are fed to the
// automaton as the extra "identity" symbol (a column whose every entry is a self-loop), and a dead automaton is
// an explicit absorbing state that is only tested once per chunk. The aligned chunk that holds a valid unit can
// never cross a page, so the over-read of up to 7 units on either side is always mapped memory.
__device__ __forceinline__ uint32_t unit_of(const uint4& v, int k) {
    const uint32_t w = (k >> 1) == 0 ? v.x : (k >> 1) == 1 ? v.y : (k >> 1) == 2 ? v.z : v.w;
    return (k & 1) ? (w >> 16) : (w & 0xFFFFu);
}

// ------------------------------------------------------------------ K2: combined DFA, one line per thread
// Table layout: rows = states + 1 (last row = dead, absorbing), columns = classes + 1 (last column = identity),
// entries premultiplied (next_row * n_cols).
template <bool kSmemTable, typename Entry>
__global__ void __launch_bounds__(kThreads) dfa_scan_kernel(DfaDev d, const uint16_t* __restrict__ text,
                                                            const int64_t* __restrict__ line_off, int sep, int64_t n_lines,
                                                            int32_t* __restrict__ ext_id) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t* s_cls = reinterpret_cast<uint16_t*>(smem_raw);  // [128] ASCII slice of the class map
    Entry* s_trans = reinterpret_cast<Entry*>(smem_raw + 256);  // [(S+1)*(C+1)] when kSmemTable
    const Entry* __restrict__ g_trans = reinterpret_cast<const Entry*>(d.trans);
    for (int i = threadIdx.x; i < 128; i += kThreads) s_cls[i] = d.cls[i];
    const uint32_t n_cols = d.n_classes + 1, ident = d.n_classes;
    if (kSmemTable)
        for (uint32_t i = threadIdx.x; i < (d.n_states + 1) * n_cols; i += kThreads) s_trans[i] = g_trans[i];
    __syncthreads();
    const uint32_t dead = d.n_states * n_cols;
    for (int64_t line = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; line < n_lines;
         line += static_cast<int64_t>(gridDim.x) * kThreads) {
        const int64_t a = line_off[line], b = line_off[line + 1] - sep;
        uint32_t st = 0;
        int64_t q = a & ~int64_t(7);
        uint32_t lo = static_cast<uint32_t>(a - q);
        for (; q < b; q += 8) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(text + q));
            const uint32_t n = b - q < 8 ? static_cast<uint32_t>(b - q) : 8u;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t u = unit_of(v, k);
                uint32_t c = u < 128 ? s_cls[u] : __ldg(d.cls + u);
                c = (static_cast<uint32_t>(k) - lo < n - lo) ? c : ident;
                st = kSmemTable ? static_cast<uint32_t>(s_trans[st + c]) : static_cast<uint32_t>(__ldg(g_trans + st + c));
            }
            lo = 0;
            if (st == dead) break;
        }
        const int32_t e = __ldg(d.accept_first + st / n_cols);  // the dead row carries -1
        ext_id[line] = e;
    }
}

// ------------------------------------------------------------------ K4: capture automaton (TDFA), one line per thread
// Per extraction: rows = states + 1 (last = dead), columns = symbol classes + 1 (last = identity: same state, no ops).
// kRegs: size of the per-line register file — 32 (registers) for ordinary extractions, kMaxTdfaRegsBig (local memory) for
// capture automata with more tag registers than that (many groups under alternations / counted repeats)
template <int kRegs>
__global__ void __launch_bounds__(kThreads) tdfa_capture_kernel(CapDev c, const uint16_t* __restrict__ text,
                                                                const int64_t* __restrict__ line_off, int sep,
                                                                int64_t n_lines, uint32_t span_stride,
                                                                int32_t* __restrict__ ext_id, int32_t* __restrict__ spans,
                                                                const TailExt* __restrict__ skip_tails, unsigned long long* __restrict__ hist) {
    __shared__ uint16_t s_cls[128];
    for (int i = threadIdx.x; i < 128; i += kThreads) s_cls[i] = c.cls[i];
    __syncthreads();
    const uint32_t n_cols = c.n_classes + 1, ident = c.n_classes;
    for (int64_t line = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; line < n_lines;
         line += static_cast<int64_t>(gridDim.x) * kThreads) {
        const int32_t e = ext_id[line];
        int32_t* out = spans + line * span_stride;
        if (e < 0) {
            if (!skip_tails)  // (with skip_tails the bucket pass has filled the rows of the MISS lines)
                for (uint32_t s = 0; s < span_stride; ++s) out[s] = -1;
            continue;
        }
        if (skip_tails && skip_tails[e].available) continue;  // the tail walk (kernels/tailwalk.cu) owns this line
        const ExtDev x = c.ext[e];
        const int64_t a = line_off[line], b = line_off[line + 1] - sep;
        const uint32_t* __restrict__ tr = c.tdfa_trans + x.trans_off;
        const uint32_t* __restrict__ opo = c.tdfa_op_off + x.opoff_off;
        const uint16_t* __restrict__ ops = c.tdfa_ops + x.ops_off;
        int32_t regs[kRegs];
        uint32_t st = 0;
        int64_t q = a & ~int64_t(7);
        uint32_t lo = static_cast<uint32_t>(a - q);
        for (; q < b; q += 8) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(text + q));
            const uint32_t n = b - q < 8 ? static_cast<uint32_t>(b - q) : 8u;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t u = unit_of(v, k);
                uint32_t sym;
                if (u < 128) {
                    sym = s_cls[u];
                } else {
                    sym = __ldg(c.cls + u);
                    // a high surrogate followed by a low surrogate is ONE java.util.regex character
                    if ((u & 0xFC00u) == 0xD800u && q + k + 1 < b && (__ldg(text + q + k + 1) & 0xFC00u) == 0xDC00u)
                        sym = c.pair_hi_class;
                }
                sym = (static_cast<uint32_t>(k) - lo < n - lo) ? sym : ident;
                const uint32_t ent = __ldg(tr + st * n_cols + sym);
                const uint32_t ol = ent >> 16;
                if (ol) {
                    const uint32_t o0 = __ldg(opo + ol), o1 = __ldg(opo + ol + 1);
                    const int32_t pos = static_cast<int32_t>(q + k - a);
                    for (uint32_t i = o0; i < o1; ++i) {
                        const uint32_t op = __ldg(ops + i);
                        const uint32_t src = op & 0xFFu;
                        regs[op >> 8] = src == 0xFFu ? pos : regs[src];
                    }
                }
                st = ent & 0xFFFFu;
            }
            lo = 0;
            if (st == x.n_states) break;  // dead
        }
        const bool ok = __ldg(c.tdfa_accepting + x.acc_off + st) != 0;  // the dead row is not accepting
        if (!ok) {
            ext_id[line] = -2 - e;
            if (hist) {  // the histogram was taken before the capture pass: move the line's count
                atomicAdd(hist + e, ~0ull);
                atomicAdd(hist + c.n_ext + 1, 1ull);
            }
            for (uint32_t s = 0; s < span_stride; ++s) out[s] = -1;
            continue;
        }
        const uint8_t* __restrict__ fin = c.tdfa_fin + x.fin_off + st * x.n_slots;
        const int32_t len = static_cast<int32_t>(b - a);
        for (uint32_t s = 0; s < x.n_slots; ++s) {
            const uint32_t f = __ldg(fin + s);
            out[s] = f == 0xFFu ? -1 : (f == 0xFEu ? len : regs[f]);
        }
        for (uint32_t s = x.n_slots; s < span_stride; ++s) out[s] = -1;
    }
}

// ------------------------------------------------------------------ K3: histogram by extraction id
constexpr int kHistSmemBins = 2048;

__global__ void __launch_bounds__(kThreads) histogram_kernel(const int32_t* __restrict__ ext_id, int64_t n_lines, uint32_t n_ext,
                                                             unsigned long long* __restrict__ hist) {
    __shared__ uint32_t bins[kHistSmemBins];
    const uint32_t nb = n_ext + 2;
    const bool local = nb <= kHistSmemBins;
    if (local) {
        for (uint32_t i = threadIdx.x; i < nb; i += kThreads) bins[i] = 0;
        __syncthreads();
    }
    for (int64_t line = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; line < n_lines;
         line += static_cast<int64_t>(gridDim.x) * kThreads) {
        const int32_t e = ext_id[line];
        const uint32_t bin = e >= 0 ? static_cast<uint32_t>(e) : (e == -1 ? n_ext : n_ext + 1);
        if (local) atomicAdd(&bins[bin], 1u);
        else atomicAdd(&hist[bin], 1ull);
    }
    if (local) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < nb; i += kThreads)
            if (bins[i]) atomicAdd(&hist[i], static_cast<unsigned long long>(bins[i]));
    }
}

// dst[i] = src[i] + bias (result assembly of a pipelined batch: piece-relative line offsets -> batch offsets)
__global__ void __launch_bounds__(kThreads) bias_copy_kernel(int64_t* __restrict__ dst, const int64_t* __restrict__ src, int64_t n, int64_t bias) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * kThreads)
        dst[i] = src[i] + bias;
}

__global__ void accumulate_kernel(int64_t* __restrict__ dst, const int64_t* __restrict__ src, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}

// ISO-8859-1 bytes -> UTF-16 units (zero extension), 16 bytes in / 32 bytes out per thread and iteration. `dst` is 16-byte
// aligned; `src` may sit at any address (a line-aligned piece of the caller's buffer copied to a 16-byte aligned
// staging buffer starts at offset 0, so both are aligned here).
__global__ void __launch_bounds__(kThreads) widen_latin1_kernel(const uint8_t* __restrict__ src, uint16_t* __restrict__ dst, int64_t n) {
    const int64_t n16 = n / 16;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; i < n16; i += static_cast<int64_t>(gridDim.x) * kThreads) {
        const uint4 v = ld_stream(reinterpret_cast<const uint4*>(src) + i);
        uint4 lo, hi;
        lo.x = __byte_perm(v.x, 0, 0x4140), lo.y = __byte_perm(v.x, 0, 0x4342);
        lo.z = __byte_perm(v.y, 0, 0x4140), lo.w = __byte_perm(v.y, 0, 0x4342);
        hi.x = __byte_perm(v.z, 0, 0x4140), hi.y = __byte_perm(v.z, 0, 0x4342);
        hi.z = __byte_perm(v.w, 0, 0x4140), hi.w = __byte_perm(v.w, 0, 0x4342);
        reinterpret_cast<uint4*>(dst)[2 * i] = lo;
        reinterpret_cast<uint4*>(dst)[2 * i + 1] = hi;
    }
    if (blockIdx.x == 0)
        for (int64_t i = n16 * 16 + threadIdx.x; i < n; i += kThreads) dst[i] = src[i];
}

int blocks_for(int64_t n, int per_block) { return static_cast<int>((n + per_block - 1) / per_block); }

}  // namespace

void k1_count_newlines(const Launch& L, const uint16_t* text, int64_t n_units, uint32_t* tile_counts) {
    if (n_units <= 0) return;
    nl_count_kernel<<<blocks_for(n_units, kNlTile), kThreads, 0, L.stream>>>(text, n_units, tile_counts);
}

void k1_scatter_newlines(const Launch& L, const uint16_t* text, int64_t n_units, const int64_t* tile_base, int64_t* line_off) {
    if (n_units <= 0) return;
    nl_scatter_kernel<<<blocks_for(n_units, kNlTile), kThreads, 0, L.stream>>>(text, n_units, tile_base, line_off);
}

void k1_count_newlines_masks(const Launch& L, const uint16_t* text, int64_t n_units, uint32_t* tile_counts, uint32_t* masks) {
    if (n_units <= 0) return;
    nl_count_mask_kernel<<<blocks_for(n_units, kNlTile), kThreads, 0, L.stream>>>(text, n_units, tile_counts, masks);
}

void k1_scatter_masks(const Launch& L, const uint32_t* masks, int64_t n_units, const int64_t* tile_base, int64_t* line_off) {
    if (n_units <= 0) return;
    const int64_t n_tiles = (n_units + kNlTile - 1) / kNlTile;
    nl_scatter_mask_kernel<<<blocks_for(n_tiles, kThreads / 32), kThreads, 0, L.stream>>>(masks, tile_base, line_off, n_tiles);
}

void k1_finish(const Launch& L, const uint16_t* text, int64_t n_units, const int64_t* total_newlines, int64_t* line_off,
               int64_t* n_lines_out) {
    nl_finish_kernel<<<1, 1, 0, L.stream>>>(text, n_units, total_newlines, line_off, n_lines_out);
}

void scan_u32_to_i64(const Launch& L, const uint32_t* in, int64_t n, int64_t* out, int64_t* scratch) {
    const int64_t nb = n > 0 ? (n + kScanTile - 1) / kScanTile : 0;
    if (nb > 0) scan_sums_kernel<<<static_cast<int>(nb), kThreads, 0, L.stream>>>(in, n, scratch);
    scan_top_kernel<<<1, 1024, 0, L.stream>>>(scratch, nb);
    scan_apply_kernel<<<static_cast<int>(nb > 0 ? nb : 1), kThreads, 0, L.stream>>>(in, n, scratch, nb, out);
}

static int persistent_grid(const Launch& L, const void* fn, size_t smem, int64_t n_lines) {
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kThreads, smem);
    if (per_sm < 1) per_sm = 1;
    int64_t want = (n_lines + kThreads - 1) / kThreads;
    int64_t cap = static_cast<int64_t>(L.sm_count) * per_sm;  // one resident wave, grid-stride over the rest
    return static_cast<int>(want < cap ? (want > 0 ? want : 1) : cap);
}

template <bool kSmem, typename Entry>
static void launch_dfa(const Launch& L, const DfaDev& d, size_t smem, const uint16_t* text, const int64_t* line_off, int sep,
                       int64_t n_lines, int32_t* ext_id) {
    auto fn = dfa_scan_kernel<kSmem, Entry>;
    allow_max_dynamic_smem(fn);
    int g = persistent_grid(L, reinterpret_cast<const void*>(fn), smem, n_lines);
    fn<<<g, kThreads, smem, L.stream>>>(d, text, line_off, sep, n_lines, ext_id);
}

void k2_dfa_scan(const Launch& L, const DfaDev& d, const uint16_t* text, const int64_t* line_off, int sep, int64_t n_lines,
                 int32_t* ext_id) {
    if (n_lines <= 0) return;
    const size_t esz = d.wide ? 4 : 2;
    const size_t table_bytes = static_cast<size_t>(d.n_states + 1) * (d.n_classes + 1) * esz;
    const bool in_smem = table_bytes <= 96 * 1024;
    const size_t smem = 256 + (in_smem ? table_bytes : 0);
    if (!d.wide) {
        if (in_smem) launch_dfa<true, uint16_t>(L, d, smem, text, line_off, sep, n_lines, ext_id);
        else launch_dfa<false, uint16_t>(L, d, smem, text, line_off, sep, n_lines, ext_id);
    } else {
        if (in_smem) launch_dfa<true, uint32_t>(L, d, smem, text, line_off, sep, n_lines, ext_id);
        else launch_dfa<false, uint32_t>(L, d, smem, text, line_off, sep, n_lines, ext_id);
    }
}

void k4_tdfa_capture(const Launch& L, const CapDev& c, const uint16_t* text, const int64_t* line_off, int sep, int64_t n_lines,
                     uint32_t span_stride, int32_t* ext_id, int32_t* spans, const TailExt* skip_tails, unsigned long long* hist) {
    if (n_lines <= 0) return;
    if (c.max_regs <= static_cast<uint32_t>(kMaxTdfaRegs)) {
        int g = persistent_grid(L, reinterpret_cast<const void*>(tdfa_capture_kernel<kMaxTdfaRegs>), 0, n_lines);
        tdfa_capture_kernel<kMaxTdfaRegs><<<g, kThreads, 0, L.stream>>>(c, text, line_off, sep, n_lines, span_stride, ext_id, spans, skip_tails, hist);
    } else {
        int g = persistent_grid(L, reinterpret_cast<const void*>(tdfa_capture_kernel<kMaxTdfaRegsBig>), 0, n_lines);
        tdfa_capture_kernel<kMaxTdfaRegsBig><<<g, kThreads, 0, L.stream>>>(c, text, line_off, sep, n_lines, span_stride, ext_id, spans, skip_tails, hist);
    }
}

void k_bias_copy(const Launch& L, int64_t* dst, const int64_t* src, int64_t n, int64_t bias) {
    if (n <= 0) return;
    const int64_t want = (n + kThreads - 1) / kThreads, cap = static_cast<int64_t>(L.sm_count) * 8;
    bias_copy_kernel<<<static_cast<int>(want < cap ? want : cap), kThreads, 0, L.stream>>>(dst, src, n, bias);
}

void k_widen_latin1(const Launch& L, const uint8_t* src, uint16_t* dst, int64_t n) {
    if (n <= 0) return;
    const int64_t want = (n / 16 + kThreads - 1) / kThreads + 1, cap = static_cast<int64_t>(L.sm_count) * 8;
    widen_latin1_kernel<<<static_cast<int>(want < cap ? want : cap), kThreads, 0, L.stream>>>(src, dst, n);
}

void k_accumulate(const Launch& L, int64_t* dst, const int64_t* src, int n) {
    if (n <= 0) return;
    accumulate_kernel<<<(n + 255) / 256, 256, 0, L.stream>>>(dst, src, n);
}

void k3_histogram(const Launch& L, const int32_t* ext_id, int64_t n_lines, uint32_t n_ext, unsigned long long* hist) {
    if (n_lines <= 0) return;
    int g = persistent_grid(L, reinterpret_cast<const void*>(histogram_kernel), 0, n_lines);
    histogram_kernel<<<g, kThreads, 0, L.stream>>>(ext_id, n_lines, n_ext, hist);
}

}  // namespace gorp
