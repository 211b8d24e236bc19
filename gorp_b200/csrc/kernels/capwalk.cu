// K4b — capture half of the text form, bucketed by extraction (sm_100a). Stands in for
// JDKRegexpCookedExtraction.match/_constructMatch (reference jdkre/JDKRegexpCookedExtraction.java:36-59) on the lines
// the combined DFA assigned to an extraction.
//
//   bucket_plan     histogram (K3) -> bucket bases, cursors, work items (extraction e, <= kCapItemLines lines of it)
//   bucket_scatter  line ids grouped by extraction (CTA-local counting, one global atomic per CTA and non-empty
//                   bucket); rows of MISS lines are filled with -1 here
//   capwalk         one WARP per work item: all lanes run the capture automaton of the same extraction (the lanes of a
//                   warp then touch the same few table rows, so the L1 gathers stay cheap and the tables never have
//                   to fit shared memory), every lane walks one line at a time in 32-byte blocks and pulls its next
//                   line from the item when it finishes one (ballot-ranked, no atomics), so lanes stay busy
//                   whatever the line lengths are. Tag registers live in shared memory, [register][thread].
//
// Table image per extraction (engine.cu builds it from host/capture.hpp: Tdfa), rows of K = classes + 1 u32 entries
// (last column = '\n'):  [0,S) states | S..S+14 = SKIP_1..15 | S+15 = DEAD | S+16 = SLOW (trap: the block is replayed
// through the general tables) | S+17+s = FRZ(s), reached at the line's '\n' from state s, absorbing.
// Entry = (byte offset of the next row inside the extraction's table) << 6 | register slot to set to the current
// position (slot n_regs = the per-thread dummy).
#include "device_common.cuh"

namespace gorp {

namespace {

using namespace dev;

constexpr int kBucketThreads = 256;
constexpr int kBucketSeg = 4096;  // lines per CTA of the scatter pass

// ------------------------------------------------------------------ bucket plan (one CTA)
// Work items = `item_lines` consecutive entries of one bucket. With `interleave` the items are listed in order of their
// RELATIVE position inside their bucket ((j + 1/2) / items of the bucket, quantised to kPlanBins classes) instead of bucket
// by bucket: the lines of an extraction are spread over the whole text, so items with the same relative position cover the
// same stretch of text — the CTAs that work through the list at the same time then share that stretch in L2 (the 128-byte
// lines at both ends of every text line are shared with its neighbours, which belong to other buckets).
constexpr uint32_t kPlanBins = 2048;

__global__ void __launch_bounds__(1024) bucket_plan_kernel(const unsigned long long* __restrict__ hist, uint32_t n_ext,
                                                           uint32_t* __restrict__ bucket_base /* [E+1] */,
                                                           uint32_t* __restrict__ cursor /* [E] */, CapItem* __restrict__ items,
                                                           uint32_t* __restrict__ n_items_out, uint32_t* __restrict__ item_ticket,
                                                           uint32_t item_lines, uint32_t interleave) {
    __shared__ uint32_t s_item_base[kCapMaxBuckets + 1];
    __shared__ uint32_t s_base[kCapMaxBuckets + 1];
    __shared__ uint32_t s_bin[kPlanBins];
    __shared__ uint32_t s_warp[32];
    for (uint32_t e = threadIdx.x; e < n_ext; e += blockDim.x) s_base[e] = static_cast<uint32_t>(hist[e]);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0, irun = 0;
        for (uint32_t e = 0; e < n_ext; ++e) {
            const uint32_t n = s_base[e];
            s_base[e] = run;
            s_item_base[e] = irun;
            run += n;
            irun += (n + item_lines - 1) / item_lines;
        }
        s_base[n_ext] = run;
        s_item_base[n_ext] = irun;
        *n_items_out = irun;
        *item_ticket = 0;
    }
    __syncthreads();
    for (uint32_t e = threadIdx.x; e <= n_ext; e += blockDim.x) {
        bucket_base[e] = s_base[e];
        if (e < n_ext) cursor[e] = s_base[e];
    }
    const uint32_t n_items = s_item_base[n_ext];
    // item i of the bucket-by-bucket numbering: its bucket (the last one whose first item is <= i), its index inside it
    auto locate = [&](uint32_t i, uint32_t& e, uint32_t& j, uint32_t& key) {
        uint32_t lo = 0, hi = n_ext;  // first bucket whose base is > i
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (s_item_base[mid] <= i) lo = mid + 1;
            else hi = mid;
        }
        e = lo - 1;
        j = i - s_item_base[e];
        const uint32_t n = s_item_base[e + 1] - s_item_base[e];
        key = min(kPlanBins - 1u, ((2u * j + 1u) * (kPlanBins / 2u)) / n);
    };
    auto put = [&](uint32_t at, uint32_t e, uint32_t j) {
        const uint32_t b = s_base[e] + j * item_lines, b1 = s_base[e + 1];
        items[at] = CapItem{e, b, b + item_lines < b1 ? b + item_lines : b1};
    };
    if (!interleave) {
        for (uint32_t i = threadIdx.x; i < n_items; i += blockDim.x) {
            uint32_t e, j, key;
            locate(i, e, j, key);
            put(i, e, j);
        }
        return;
    }
    for (uint32_t k = threadIdx.x; k < kPlanBins; k += blockDim.x) s_bin[k] = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n_items; i += blockDim.x) {
        uint32_t e, j, key;
        locate(i, e, j, key);
        atomicAdd(&s_bin[key], 1u);
    }
    __syncthreads();
    {  // exclusive scan of the kPlanBins counts: two bins per thread (blockDim.x == 1024)
        const uint32_t c0 = s_bin[2 * threadIdx.x], c1 = s_bin[2 * threadIdx.x + 1];
        uint32_t incl = c0 + c1;
        const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= static_cast<uint32_t>(o)) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint32_t wbase = 0;
        for (uint32_t w = 0; w < warp; ++w) wbase += s_warp[w];
        s_bin[2 * threadIdx.x] = wbase + incl - c0 - c1;
        s_bin[2 * threadIdx.x + 1] = wbase + incl - c1;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n_items; i += blockDim.x) {
        uint32_t e, j, key;
        locate(i, e, j, key);
        put(atomicAdd(&s_bin[key], 1u), e, j);
    }
}

// ------------------------------------------------------------------ bucket scatter
__global__ void __launch_bounds__(kBucketThreads) bucket_scatter_kernel(const int32_t* __restrict__ ext_id, int64_t n_lines, uint32_t n_ext,
                                                                        uint32_t* __restrict__ cursor, uint32_t* __restrict__ perm,
                                                                        int32_t* __restrict__ spans, uint32_t span_stride,
                                                                        const int64_t* __restrict__ line_off, LineRec* __restrict__ recs, int sep,
                                                                        const TailExt* __restrict__ tails) {
    __shared__ uint32_t s_cnt[kCapMaxBuckets];
    __shared__ uint32_t s_pos[kCapMaxBuckets];
    __shared__ uint8_t s_perm_needed[kCapMaxBuckets];  // 0: the extraction's lines go to the tail walk, which reads records only
    for (uint32_t i = threadIdx.x; i < n_ext; i += kBucketThreads) s_perm_needed[i] = (!recs || !tails[i].available) ? 1 : 0;
    for (int64_t seg0 = static_cast<int64_t>(blockIdx.x) * kBucketSeg; seg0 < n_lines; seg0 += static_cast<int64_t>(gridDim.x) * kBucketSeg) {
        for (uint32_t i = threadIdx.x; i < n_ext; i += kBucketThreads) s_cnt[i] = 0;
        __syncthreads();
        const int64_t seg1 = seg0 + kBucketSeg < n_lines ? seg0 + kBucketSeg : n_lines;
        int32_t mine[kBucketSeg / kBucketThreads];
        uint32_t rank[kBucketSeg / kBucketThreads];
#pragma unroll
        for (int k = 0; k < kBucketSeg / kBucketThreads; ++k) {
            const int64_t line = seg0 + k * kBucketThreads + threadIdx.x;
            mine[k] = line < seg1 ? ext_id[line] : -1;
            rank[k] = mine[k] >= 0 ? atomicAdd(&s_cnt[mine[k]], 1u) : 0u;
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n_ext; i += kBucketThreads) {
            const uint32_t n = s_cnt[i];
            s_pos[i] = n ? atomicAdd(cursor + i, n) : 0u;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kBucketSeg / kBucketThreads; ++k) {
            const int64_t line = seg0 + k * kBucketThreads + threadIdx.x;
            if (line >= seg1) continue;
            if (mine[k] >= 0) {
                const uint32_t at = s_pos[mine[k]] + rank[k];
                // the tail walk reads records, the bucketed capture walk (extractions without a tail) reads `perm`
                if (s_perm_needed[mine[k]]) perm[at] = static_cast<uint32_t>(line);
                if (recs) {  // start, id and length of the line in one record (kernels/tailwalk.cu)
                    const int64_t a = line_off[line], len = line_off[line + 1] - sep - a;
                    const int4 r = make_int4(static_cast<int>(static_cast<uint64_t>(a) & 0xFFFFFFFFu), static_cast<int>(static_cast<uint64_t>(a) >> 32),
                                             static_cast<int>(line), static_cast<int>(len > 0xFFFFFFFFll ? 0xFFFFFFFFll : len));
                    *reinterpret_cast<int4*>(recs + at) = r;
                }
            } else {  // MISS: the row is all -1
                int32_t* out = spans + line * span_stride;
                for (uint32_t s = 0; s < span_stride; ++s) out[s] = -1;
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ capture walk
__device__ __forceinline__ uint32_t ldg32_off(const unsigned char* __restrict__ base, uint32_t off) {
    return __ldg(reinterpret_cast<const uint32_t*>(base + off));
}

// kSmemTab: the extraction's table was copied to shared memory (tab_abs); otherwise it is read through L1/L2 (tab)
template <bool kSmemTab, int kByte>
__device__ __forceinline__ void cw_step(uint32_t& st, uint32_t& fin, uint32_t dead_off, uint32_t w, uint32_t cls_abs, uint32_t tab_abs,
                                        const unsigned char* __restrict__ tab, uint32_t reg_abs, uint32_t reg_stride, uint32_t pos) {
    uint32_t b, a;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(b) : "r"(w), "n"(kByte == 0 ? 0x4440 : 0x4442));
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(a) : "r"(b), "r"(cls_abs));
    const uint32_t c4 = lds32(a);
    uint32_t ent;
    if (kSmemTab) {  // the shared-memory copy has no FRZ rows: ids beyond DEAD read the DEAD row, `fin` keeps the highest id seen
        ent = lds32(tab_abs + min(st, dead_off) + c4);
    } else {
        ent = ldg32_off(tab, st + c4);
    }
    st = ent >> 6;
    if (kSmemTab) fin = max(fin, st);
    uint32_t sa;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(sa) : "r"(ent & 63u), "r"(reg_stride), "r"(reg_abs));
    sts32(sa, pos);
}

// one step on ANY unit (blocks that hold a unit >= 0x80): the class comes from the full class map, a high surrogate that
// is followed by a low surrogate takes the PAIR_HI class (java.util.regex consumes the pair as one character)
template <bool kSmemTab>
__device__ __forceinline__ void cw_step_any(uint32_t& st, uint32_t& fin, uint32_t dead_off, uint32_t u, uint32_t nx, const CapDev& c,
                                            uint32_t cls_abs, uint32_t tab_abs, const unsigned char* __restrict__ tab, uint32_t reg_abs,
                                            uint32_t reg_stride, uint32_t pos) {
    uint32_t c4;
    if (u < 0x80u) {
        c4 = lds32(cls_abs + u * 4);
    } else {
        c4 = 4u * __ldg(c.cls + u);
        if ((u & 0xFC00u) == 0xD800u && (nx & 0xFC00u) == 0xDC00u) c4 = 4u * c.pair_hi_class;
    }
    uint32_t ent;
    if (kSmemTab) {
        ent = lds32(tab_abs + min(st, dead_off) + c4);
    } else {
        ent = ldg32_off(tab, st + c4);
    }
    st = ent >> 6;
    if (kSmemTab) fin = max(fin, st);
    sts32(reg_abs + (ent & 63u) * reg_stride, pos);
}

// 16 units through the general tables (units >= 0x80, surrogate pairs, transitions with several register commands).
// `q` = text position of the block, `a` = text position of the line start; units at or beyond n_units read as '\n'.
// `st` is a row byte offset of the extraction's image on entry and exit.
__device__ __noinline__ uint32_t cw_slow16(const CapDev& c, const ExtDev& x, const CapImgExt& fx, uint32_t st,
                                           const uint16_t* __restrict__ text, int64_t q, int64_t a, int64_t n_units, uint32_t reg_abs,
                                           uint32_t reg_stride) {
    const uint32_t S = fx.n_states;
    uint32_t row = st / fx.row_bytes;
    const uint32_t n_cols = c.n_classes + 1;
    const uint32_t* __restrict__ tr = c.tdfa_trans + x.trans_off;
    const uint32_t* __restrict__ opo = c.tdfa_op_off + x.opoff_off;
    const uint16_t* __restrict__ ops = c.tdfa_ops + x.ops_off;
#pragma unroll 1
    for (int k = 0; k < 16; ++k) {
        if (row >= S + 15) break;  // DEAD / FRZ
        const int64_t p = q + k;
        const uint32_t u = p < n_units ? __ldg(text + p) : 0x0Au;
        if (row >= S) {  // SKIP_j
            row = row == S ? 0u : row - 1;
            continue;
        }
        if (u == 0x0Au) {
            row = S + 17 + row;
            break;
        }
        const uint32_t pos = static_cast<uint32_t>(p - a);
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
        if (row == S) row = S + 15;  // the general table's dead row index is S
    }
    return row * fx.row_bytes;
}

// One work item (lines of one extraction) walked by all warps of the CTA: lanes claim lines from the CTA's cursor.
template <bool kSmemTab>
__device__ __forceinline__ void cw_item(const CapWalkParams& P, const CapItem& it, uint32_t* s_cursor, uint4* s_fin, uint32_t cls_abs,
                                        uint32_t tab_abs, uint32_t reg_abs, uint32_t reg_abs_warp, uint32_t lane) {
    const uint32_t e = it.ext;
    const CapImgExt fx = P.img.ext[e];
    const ExtDev x = P.cap.ext[e];
    const unsigned char* __restrict__ tab = reinterpret_cast<const unsigned char*>(P.img.image) + fx.tab_off;
    const uint32_t reg_stride = kCapWalkThreads * 4;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t stride = P.span_stride;
    // i / stride == __umulhi(i, inv_stride) for every i < 2048 and stride <= 62 (checked exhaustively; a 16-bit reciprocal
    // is not enough for i < 32 * stride: it is one too high from i = 1679 on for stride 56, 1499 for 60, 1115 for 62)
    const uint32_t inv_stride = 0xFFFFFFFFu / stride + 1u;
    bool exhausted = false;  // warp-uniform: the item has no unclaimed line left

    // per-lane state: the line being walked, and the NEXT line of the lane, claimed one line ahead so that its id
    // (perm), start and end (line_off) are loaded long before they are needed
    bool active = false;
    uint32_t line = 0, len = 0;
    int64_t a = 0, q = 0;
    uint32_t st = fx.dead_off;
    uint32_t nstage = 0;  // 0 = no next line, 1 = id requested, 2 = start and end requested
    uint32_t nline = 0;
    int64_t na = 0, nb = 0;
    for (;;) {
        if (!active && nstage) {  // start the claimed line
            if (nstage == 1) {
                na = __ldg(P.line_off + nline);
                nb = __ldg(P.line_off + nline + 1);
            }
            line = nline;
            a = na;
            len = static_cast<uint32_t>(nb - 1 - na);
            q = a & ~int64_t(15);
            const uint32_t lo = static_cast<uint32_t>(a - q);
            st = lo ? (fx.n_states + lo - 1) * fx.row_bytes : 0u;
            active = true;
            nstage = 0;
        } else if (nstage == 1) {
            na = __ldg(P.line_off + nline);
            nb = __ldg(P.line_off + nline + 1);
            nstage = 2;
        }
        if (!exhausted) {  // lanes without a next line claim the next entries of the item
            const uint32_t want = __ballot_sync(0xffffffffu, nstage == 0);
            if (want) {
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(s_cursor, static_cast<uint32_t>(__popc(want)));
                base = __shfl_sync(0xffffffffu, base, 0);
                const uint32_t idx = base + static_cast<uint32_t>(__popc(want & lt_mask));
                if (nstage == 0 && idx < it.end) {
                    nline = __ldg(P.perm + idx);
                    nstage = 1;
                }
                exhausted = base + static_cast<uint32_t>(__popc(want)) >= it.end;
            }
        }
        if (!__any_sync(0xffffffffu, active || nstage != 0)) break;
        bool finished = false;
        if (active) {
            const Units16 u = P.flags & 1u ? load_units16(P.text, q, P.n_units) : load_units16_l2keep(P.text, q, P.n_units);
            const uint32_t st0 = st;
            uint32_t fin = 0;
            const uint32_t pos = static_cast<uint32_t>(q - a);  // negative while skipping: only ever stored to the dummy register
            if (((u.a.x | u.a.y | u.a.z | u.a.w | u.b.x | u.b.y | u.b.z | u.b.w) & 0xFF80FF80u) == 0u) {
                cw_step<kSmemTab, 0>(st, fin, fx.dead_off, u.a.x, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos);
                cw_step<kSmemTab, 2>(st, fin, fx.dead_off, u.a.x, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 1);
                cw_step<kSmemTab, 0>(st, fin, fx.dead_off, u.a.y, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 2);
                cw_step<kSmemTab, 2>(st, fin, fx.dead_off, u.a.y, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 3);
                cw_step<kSmemTab, 0>(st, fin, fx.dead_off, u.a.z, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 4);
                cw_step<kSmemTab, 2>(st, fin, fx.dead_off, u.a.z, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 5);
                cw_step<kSmemTab, 0>(st, fin, fx.dead_off, u.a.w, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 6);
                cw_step<kSmemTab, 2>(st, fin, fx.dead_off, u.a.w, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 7);
                cw_step<kSmemTab, 0>(st, fin, fx.dead_off, u.b.x, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 8);
                cw_step<kSmemTab, 2>(st, fin, fx.dead_off, u.b.x, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 9);
                cw_step<kSmemTab, 0>(st, fin, fx.dead_off, u.b.y, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 10);
                cw_step<kSmemTab, 2>(st, fin, fx.dead_off, u.b.y, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 11);
                cw_step<kSmemTab, 0>(st, fin, fx.dead_off, u.b.z, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 12);
                cw_step<kSmemTab, 2>(st, fin, fx.dead_off, u.b.z, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 13);
                cw_step<kSmemTab, 0>(st, fin, fx.dead_off, u.b.w, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 14);
                cw_step<kSmemTab, 2>(st, fin, fx.dead_off, u.b.w, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + 15);
                if (kSmemTab && fin >= fx.dead_off) st = fin;  // SLOW and FRZ ids do not survive the steps that follow them
                if (st == fx.slow_off) st = cw_slow16(P.cap, x, fx, st0, P.text, q, a, P.n_units, reg_abs, reg_stride);
            } else {  // a unit >= 0x80 in the block: same tables, classes through the full class map
                const uint32_t w[8] = {u.a.x, u.a.y, u.a.z, u.a.w, u.b.x, u.b.y, u.b.z, u.b.w};
                // the unit after the block: only a high surrogate in the block's last unit looks at it; units at or beyond
                // n_units read as '\n' (the pair test of the general path: p + 1 < n_units)
                const uint32_t after = ((w[7] >> 16) & 0xFC00u) == 0xD800u && q + 16 < P.n_units ? __ldg(P.text + q + 16) : 0x0Au;
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const uint32_t cu = (k & 1) ? (w[k >> 1] >> 16) : (w[k >> 1] & 0xFFFFu);
                    const uint32_t nu = k == 15 ? after : ((k & 1) ? (w[(k + 1) >> 1] & 0xFFFFu) : (w[k >> 1] >> 16));
                    cw_step_any<kSmemTab>(st, fin, fx.dead_off, cu, nu, P.cap, cls_abs, tab_abs, tab, reg_abs, reg_stride, pos + k);
                }
                if (kSmemTab && fin >= fx.dead_off) st = fin;
                if (st == fx.slow_off) st = cw_slow16(P.cap, x, fx, st0, P.text, q, a, P.n_units, reg_abs, reg_stride);
            }
            q += 16;
            finished = st >= fx.dead_off;  // DEAD (rejected) or FRZ(s)
        }
        uint32_t fmeta = 0xFFFFFFFFu;  // final capture state of an accepted line
        if (finished) {
            active = false;
            if (st >= fx.frz_off) {
                const uint32_t s = (st - fx.frz_off) / fx.row_bytes;
                if (__ldg(P.cap.tdfa_accepting + x.acc_off + s) != 0) fmeta = s;
            }
        }
        // result rows of the lines that ended in this iteration, written by the whole warp: the finished lanes post
        // (line, final state, length, lane) in the warp's staging area, then lane i writes entry i % stride of row i / stride
        const uint32_t fin_mask = __ballot_sync(0xffffffffu, finished);
        if (fin_mask) {
            if (finished) {
                s_fin[__popc(fin_mask & lt_mask)] = make_uint4(line, fmeta, len, lane);
                if (fmeta == 0xFFFFFFFFu) {  // the combined DFA accepted, java.util.regex does not (Gorp.java:173-177)
                    P.ext_id[line] = -2 - static_cast<int32_t>(e);
                    atomicAdd(P.hist + e, ~0ull);  // -1
                    atomicAdd(P.hist + P.cap.n_ext + 1, 1ull);
                }
            }
            __syncwarp();  // staging area and the finished lanes' tag registers are read by the other lanes
            const uint32_t total = static_cast<uint32_t>(__popc(fin_mask)) * stride;
            for (uint32_t i = lane; i < total; i += 32) {
                const uint32_t j = __umulhi(i, inv_stride), k = i - j * stride;
                const uint4 f = s_fin[j];
                int32_t val = -1;
                if (f.y != 0xFFFFFFFFu && k < x.n_slots) {
                    const uint32_t r = __ldg(P.cap.tdfa_fin + x.fin_off + f.y * x.n_slots + k);
                    if (r == 0xFEu) val = static_cast<int32_t>(f.z);
                    else if (r != 0xFFu) val = static_cast<int32_t>(lds32(reg_abs_warp + f.w * 4 + r * reg_stride));
                }
                P.spans[static_cast<int64_t>(f.x) * stride + k] = val;
            }
            __syncwarp();  // the staging area is rewritten in the next iteration
        }
    }
}

__global__ void __launch_bounds__(kCapWalkThreads, 4) capwalk_kernel(CapWalkParams P) {
    extern __shared__ __align__(16) uint32_t s_mem[];  // [cls128][registers: (n_regs + 1) x blockDim][table of the item]
    __shared__ uint32_t s_item, s_cursor, s_loaded;
    __shared__ uint4 s_fin_all[kCapWalkThreads];  // per warp: the lines that finished in the current iteration
    for (uint32_t i = threadIdx.x; i < 128; i += kCapWalkThreads) s_mem[i] = __ldg(P.img.cls128 + i);
    if (threadIdx.x == 0) s_loaded = 0xFFFFFFFFu;
    const uint32_t cls_abs = static_cast<uint32_t>(__cvta_generic_to_shared(s_mem));
    const uint32_t reg_abs = cls_abs + 512 + threadIdx.x * 4;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t reg_abs_warp = reg_abs - lane * 4;  // registers of lane 0 of this warp
    const uint32_t tab_words0 = 128 + (P.img.n_regs + 1) * kCapWalkThreads;
    const uint32_t tab_abs = cls_abs + tab_words0 * 4;
    const uint32_t n_items = *P.n_items;
    for (;;) {
        __syncthreads();  // the previous item is finished (its table and s_item / s_cursor are free)
        if (threadIdx.x == 0) s_item = atomicAdd(P.item_ticket, 1u);
        __syncthreads();
        const uint32_t item = s_item;
        if (item >= n_items) break;
        const CapItem it = P.items[item];
        if (P.skip_tails && P.skip_tails[it.ext].available) continue;  // the tail walk (kernels/tailwalk.cu) takes this item
        const CapImgExt fx = P.img.ext[it.ext];
        // the extraction's table goes to shared memory when it fits: a warp-wide gather through L1 is as slow as its
        // slowest lane (one L1 miss among 32 lanes costs the whole warp an L2 round trip), LDS has no such tail
        const uint32_t tab_bytes = fx.frz_off;  // (S + 17) rows: states, SKIP, DEAD, SLOW (the FRZ rows stay behind)
        const bool in_smem = tab_bytes <= P.smem_table_bytes;
        if (in_smem && s_loaded != it.ext) {
            const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(P.img.image) + fx.tab_off);
            uint4* dst = reinterpret_cast<uint4*>(s_mem + tab_words0);
            for (uint32_t i = threadIdx.x; i < (tab_bytes + 15) / 16; i += kCapWalkThreads) dst[i] = __ldg(src + i);
        }
        if (threadIdx.x == 0) s_cursor = it.begin;
        __syncthreads();
        if (threadIdx.x == 0 && in_smem) s_loaded = it.ext;
        uint4* s_fin = s_fin_all + (threadIdx.x & ~31u);
        if (in_smem) cw_item<true>(P, it, &s_cursor, s_fin, cls_abs, tab_abs, reg_abs, reg_abs_warp, lane);
        else cw_item<false>(P, it, &s_cursor, s_fin, cls_abs, tab_abs, reg_abs, reg_abs_warp, lane);
    }
}

}  // namespace

void k4b_bucket(const Launch& L, const int32_t* ext_id, int64_t n_lines, uint32_t n_ext, const unsigned long long* hist,
                uint32_t* bucket_base, uint32_t* cursor, uint32_t* perm, CapItem* items, uint32_t* n_items, uint32_t* item_ticket,
                int32_t* spans, uint32_t span_stride, const int64_t* line_off, LineRec* recs, int sep, const TailExt* tails,
                uint32_t item_lines, bool interleave) {
    if (item_lines < 32 || item_lines > kCapItemLines) item_lines = kCapItemLines;
    bucket_plan_kernel<<<1, 1024, 0, L.stream>>>(hist, n_ext, bucket_base, cursor, items, n_items, item_ticket, item_lines, interleave ? 1u : 0u);
    if (n_lines <= 0) return;
    const int64_t want = (n_lines + kBucketSeg - 1) / kBucketSeg, cap = static_cast<int64_t>(L.sm_count) * 8;
    bucket_scatter_kernel<<<static_cast<int>(want < cap ? want : cap), kBucketThreads, 0, L.stream>>>(ext_id, n_lines, n_ext, cursor, perm, spans,
                                                                                                     span_stride, line_off, recs, sep, tails);
}

size_t capwalk_smem_bytes(const CapImgDev& img) {
    return 512 + static_cast<size_t>(img.n_regs + 1) * kCapWalkThreads * 4 + img.smem_table_bytes;
}

void k4b_capwalk(const Launch& L, const CapWalkParams& P) {
    const size_t smem = capwalk_smem_bytes(P.img);
    allow_max_dynamic_smem(capwalk_kernel);
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, capwalk_kernel, kCapWalkThreads, smem);
    if (per_sm < 1) per_sm = 1;
    capwalk_kernel<<<L.sm_count * per_sm, kCapWalkThreads, smem, L.stream>>>(P);
}

}  // namespace gorp
