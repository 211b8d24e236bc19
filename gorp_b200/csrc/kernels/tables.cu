// Value tables of a device-resident result (gorp_extract_tables_device, DESIGN.md §5.5): the matched lines partitioned
// stably by extraction, then per group one Arrow-layout string column (64-bit offsets, validity bitmap, the values
// gathered from the caller's text).
//   count   : per tile of lines, lines per extraction          -> counts[e * n_tiles + t]
//   scan    : scan_u32_to_i64 over counts (extraction-major)   -> start of every (extraction, tile) in its table
//   layout  : one CTA, every buffer position of every table     -> TableLayout[E + 1]
//   scatter : the tile walked again, lines ranked inside it     -> row indexes
//   len     : 256 rows of a table per task: u32 lengths, validity words, per-column totals and null counts
//   (host: the per-column totals size the data) scan over every column's lengths at once -> offsets
//   gather  : 32 rows of a column per task: offsets rebased in place, values copied with 16-byte stores
//   rebase  : (host calls on several devices) a device's row indexes and offsets plus its bases, its bitmaps shifted to
//             the bit position of its first row -> one table per extraction across the devices
#include "kernels.cuh"

namespace gorp {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int64_t kLenRows = 256;  // rows of a table per task of the length pass

__device__ __forceinline__ int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// partition key of line i: its extraction, -1 for MISS / CAPTURE_FAIL / past the tile
__device__ __forceinline__ int line_key(const int32_t* ext_id, int64_t i, int64_t end) { return i < end ? max(ext_id[i], -1) : -1; }

// warps per CTA of the tile passes: every warp keeps one counter per extraction in shared memory (<= 32 KB a CTA)
int tile_warps(uint32_t n_ext) { return n_ext <= 1024 ? 4 : 1; }

// One warp per tile. Lanes of one extraction find each other with __match_any_sync; the lowest of them counts for all.
__global__ void tables_count_kernel(const int32_t* __restrict__ ext_id, int64_t n, uint32_t n_ext, int64_t tile_lines, int64_t n_tiles,
                                    uint32_t* __restrict__ counts) {
    extern __shared__ uint32_t s_cnt[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    if (t >= n_tiles) return;
    uint32_t* cnt = s_cnt + static_cast<size_t>(warp) * n_ext;
    for (uint32_t e = lane; e < n_ext; e += 32) cnt[e] = 0;
    __syncwarp();
    const int64_t i0 = t * tile_lines, i1 = min(i0 + tile_lines, n);
    for (int64_t i = i0; i < i1; i += 32) {
        const int e = line_key(ext_id, i + lane, i1);
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, e);
        if (e >= 0 && lane == __ffs(peers) - 1) cnt[e] += __popc(peers);
        __syncwarp();
    }
    for (uint32_t e = lane; e < n_ext; e += 32) counts[static_cast<int64_t>(e) * n_tiles + t] = cnt[e];
}

// Rows of table e = starts[(e+1) * n_tiles] - starts[e * n_tiles]; every position is laid out from those counts (thread 0
// in shared memory: E <= kCapMaxBuckets). Entry E holds the totals.
__global__ void tables_layout_kernel(const int64_t* __restrict__ starts, int64_t n_tiles, uint32_t n_ext, const uint32_t* __restrict__ slots,
                                     uint32_t with_groups, TableLayout* __restrict__ lay) {
    extern __shared__ int64_t s_rows[];
    uint32_t* s_cols = reinterpret_cast<uint32_t*>(s_rows + n_ext);
    for (uint32_t e = threadIdx.x; e < n_ext; e += blockDim.x) {
        s_rows[e] = starts[static_cast<int64_t>(e + 1) * n_tiles] - starts[static_cast<int64_t>(e) * n_tiles];
        s_cols[e] = with_groups ? slots[e] / 2 : 0;
    }
    __syncthreads();
    if (threadIdx.x) return;
    TableLayout acc{};
    for (uint32_t e = 0; e < n_ext; ++e) {
        TableLayout x = acc;
        x.n_rows = s_rows[e];
        x.n_cols = s_cols[e];
        x.seg = round_up(x.n_rows + 1, 8);
        x.vwords = round_up((x.n_rows + 31) / 32, 16);
        lay[e] = x;
        acc.row_base += round_up(x.n_rows, 8);
        acc.off_base += x.n_cols * x.seg;
        acc.valid_base += x.n_cols * x.vwords;
        acc.len_task += x.n_cols ? (x.seg + kLenRows - 1) / kLenRows : 0;
        acc.gather_task += x.n_cols * (x.n_rows / 32 + 1);
        acc.col_base += x.n_cols;
        acc.n_rows += x.n_rows;
    }
    lay[n_ext] = acc;
}

// The tiles of the count pass again: a line's row is the start of (its extraction, this tile), plus the lines of that
// extraction before it in the tile (earlier 32-line steps, then lower lanes): the partition keeps line order.
__global__ void tables_scatter_kernel(const int32_t* __restrict__ ext_id, int64_t n, uint32_t n_ext, int64_t tile_lines, int64_t n_tiles,
                                      const int64_t* __restrict__ starts, const TableLayout* __restrict__ lay, int64_t* __restrict__ rows) {
    extern __shared__ int64_t s_pos[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    if (t >= n_tiles) return;
    int64_t* pos = s_pos + static_cast<size_t>(warp) * n_ext;
    for (uint32_t e = lane; e < n_ext; e += 32)
        pos[e] = lay[e].row_base + starts[static_cast<int64_t>(e) * n_tiles + t] - starts[static_cast<int64_t>(e) * n_tiles];
    __syncwarp();
    const unsigned below = (1u << lane) - 1;
    const int64_t i0 = t * tile_lines, i1 = min(i0 + tile_lines, n);
    for (int64_t i = i0; i < i1; i += 32) {
        const int e = line_key(ext_id, i + lane, i1);
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, e);
        if (e >= 0) rows[pos[e] + __popc(peers & below)] = i + lane;
        __syncwarp();
        if (e >= 0 && lane == __ffs(peers) - 1) pos[e] += __popc(peers);
        __syncwarp();
    }
}

// the table whose tasks contain `task`: the last e with first[e] <= task (tables without tasks share their successor's
// first task and are never the last such e)
template <class F>
__device__ __forceinline__ uint32_t table_of(int64_t task, uint32_t n_ext, F first) {
    uint32_t lo = 0, hi = n_ext - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (first(mid) <= task) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// One warp per task of 256 rows of a table: each row's span row is read once for all its columns. Writes the u32 length
// of every entry of the table's offset segments (0 for the entries past the last row), one validity word per 32 rows, and
// adds the column totals and null counts (stats[2 * col], stats[2 * col + 1]) once per task.
__global__ void __launch_bounds__(kThreads) tables_len_kernel(const TableLayout* __restrict__ lay, uint32_t n_ext, const int64_t* __restrict__ rows,
                                                              const int32_t* __restrict__ spans, uint32_t stride, uint32_t* __restrict__ lens,
                                                              uint32_t* __restrict__ valid, unsigned long long* __restrict__ stats) {
    __shared__ unsigned long long s_tot[kWarps][32], s_null[kWarps][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n_tasks = lay[n_ext].len_task;
    for (int64_t task = static_cast<int64_t>(blockIdx.x) * kWarps + warp; task < n_tasks; task += static_cast<int64_t>(gridDim.x) * kWarps) {
        const TableLayout L = lay[table_of(task, n_ext, [&](uint32_t e) { return lay[e].len_task; })];
        const int64_t r0 = (task - L.len_task) * kLenRows;
        s_tot[warp][lane] = 0;
        s_null[warp][lane] = 0;
        __syncwarp();
        for (int64_t rb = r0; rb < r0 + kLenRows && rb < L.seg; rb += 32) {
            const int64_t r = rb + lane;
            const bool in = r < L.n_rows;
            const unsigned in_mask = __ballot_sync(0xFFFFFFFFu, in);
            const int32_t* row = in ? spans + rows[L.row_base + r] * stride : nullptr;
            for (uint32_t k = 0; k < L.n_cols; ++k) {
                const int2 st = in ? *reinterpret_cast<const int2*>(row + 2 * k) : make_int2(-1, -1);
                const bool ok = st.x >= 0;
                const uint32_t len = ok ? static_cast<uint32_t>(st.y - st.x) : 0u;
                const int64_t seg = L.off_base + k * L.seg;
                if (r < L.seg) lens[seg + r] = len;
                const unsigned ok_mask = __ballot_sync(0xFFFFFFFFu, ok);
                // (two 16-bit halves: 32 lengths of up to 2^31 units overflow one u32 sum)
                const unsigned lo = __reduce_add_sync(0xFFFFFFFFu, len & 0xFFFFu), hi = __reduce_add_sync(0xFFFFFFFFu, len >> 16);
                if (lane == 0) {
                    if (rb < L.n_rows) valid[L.valid_base + k * L.vwords + rb / 32] = ok_mask;
                    s_null[warp][k] += __popc(in_mask & ~ok_mask);
                    s_tot[warp][k] += lo + (static_cast<unsigned long long>(hi) << 16);
                }
            }
        }
        __syncwarp();
        if (lane < static_cast<int>(L.n_cols)) {
            const int64_t col = L.col_base + lane;
            if (s_tot[warp][lane]) atomicAdd(&stats[2 * col], s_tot[warp][lane]);
            if (s_null[warp][lane]) atomicAdd(&stats[2 * col + 1], s_null[warp][lane]);
        }
        __syncwarp();
    }
}

// One warp per task of 32 rows of one column (a column of n rows has n / 32 + 1 tasks: the last one also writes offset
// entry n). The destination range of the 32 rows is contiguous: the warp fills its aligned 16-byte blocks with vector
// stores and the units outside them one by one. The unit at destination u belongs to the last row whose offset is <= u;
// the rows' offsets and source starts sit in shared memory, so a lane finds it by binary search once per block and steps
// forward from there.
template <class T>
__global__ void __launch_bounds__(kThreads) tables_gather_kernel(const TableLayout* __restrict__ lay, uint32_t n_ext, const int64_t* __restrict__ rows,
                                                                 const int64_t* __restrict__ line_off, const int32_t* __restrict__ spans, uint32_t stride,
                                                                 const T* __restrict__ text, const uint32_t* __restrict__ lens, int64_t* __restrict__ offs,
                                                                 const int64_t* __restrict__ col_info, uint8_t* __restrict__ data) {
    constexpr int V = 16 / sizeof(T);
    __shared__ int64_t s_dst[kWarps][32], s_src[kWarps][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t* dst_of = s_dst[warp];
    int64_t* src_of = s_src[warp];
    const int64_t n_tasks = lay[n_ext].gather_task;
    for (int64_t task = static_cast<int64_t>(blockIdx.x) * kWarps + warp; task < n_tasks; task += static_cast<int64_t>(gridDim.x) * kWarps) {
        const TableLayout L = lay[table_of(task, n_ext, [&](uint32_t e) { return lay[e].gather_task; })];
        const int64_t per_col = L.n_rows / 32 + 1, rel = task - L.gather_task;
        const int64_t k = rel / per_col, r0 = (rel % per_col) * 32;
        const int64_t col = L.col_base + k;
        const int64_t flat_base = col_info[2 * col];
        T* out = reinterpret_cast<T*>(data + col_info[2 * col + 1]);
        int64_t* o = offs + L.off_base + k * L.seg;
        const int64_t r = r0 + lane;
        int64_t dst = 0, src = 0;
        uint32_t len = 0;
        if (r <= L.n_rows) {
            dst = o[r] - flat_base;
            o[r] = dst;  // (entry r belongs to this task only)
        }
        if (r < L.n_rows) {
            len = lens[L.off_base + k * L.seg + r];
            if (len) {
                const int64_t line = rows[L.row_base + r];
                src = line_off[line] + spans[line * stride + 2 * k];
            }
        }
        const int nr = static_cast<int>(min(static_cast<int64_t>(32), L.n_rows - r0));
        if (nr <= 0) continue;
        const int64_t d0 = __shfl_sync(0xFFFFFFFFu, dst, 0), d1 = __shfl_sync(0xFFFFFFFFu, dst + len, nr - 1);
        dst_of[lane] = lane < nr ? dst : d1;
        src_of[lane] = src;
        __syncwarp();
        auto find = [&](int64_t u) {
            int lo = 0, hi = nr - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (dst_of[mid] <= u) lo = mid;
                else hi = mid - 1;
            }
            return lo;
        };
        auto unit = [&](int64_t u, int& j) -> T {
            while (j + 1 < nr && dst_of[j + 1] <= u) ++j;
            return text[src_of[j] + (u - dst_of[j])];
        };
        const int64_t a0 = (d0 + V - 1) / V, a1 = d1 / V;  // whole 16-byte blocks [a0, a1)
        for (int64_t v = a0 + lane; v < a1; v += 32) {
            int j = find(v * V);
            union {
                uint4 q;
                T u[V];
            } b;
#pragma unroll
            for (int x = 0; x < V; ++x) b.u[x] = unit(v * V + x, j);
            reinterpret_cast<uint4*>(out)[v] = b.q;
        }
        const int64_t head_end = a0 < a1 ? a0 * V : d1, tail_begin = a0 < a1 ? a1 * V : d1;
        for (int64_t u = d0 + lane; u < head_end; u += 32) {
            int j = find(u);
            out[u] = unit(u, j);
        }
        for (int64_t u = tail_begin + lane; u < d1; u += 32) {
            int j = find(u);
            out[u] = unit(u, j);
        }
        __syncwarp();
    }
}

// One block of kRebaseBlock entries (or output bytes) of one job per iteration; the job is found by binary search over the
// jobs' first blocks, as the table of a task above.
constexpr int64_t kRebaseBlock = 8 * kThreads;
__global__ void __launch_bounds__(kThreads) tables_rebase_kernel(const RebaseJob* __restrict__ jobs, uint32_t n_jobs, int64_t n_blocks) {
    for (int64_t blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
        const RebaseJob J = jobs[table_of(blk, n_jobs, [&](uint32_t j) { return jobs[j].first_block; })];
        const int64_t i0 = (blk - J.first_block) * kRebaseBlock;
        if (!J.shift) {
            const int64_t* src = static_cast<const int64_t*>(J.src);
            int64_t* dst = static_cast<int64_t*>(J.dst);
            for (int64_t i = i0 + threadIdx.x; i < min(i0 + kRebaseBlock, J.n); i += kThreads) dst[i] = src[i] + J.add;
        } else {
            // output byte j holds input bits [8j - shift, 8j + 8 - shift): the top of byte j - 1 and the bottom of byte j
            const uint8_t* src = static_cast<const uint8_t*>(J.src);
            uint8_t* dst = static_cast<uint8_t*>(J.dst);
            const int64_t nb_in = (J.n + 7) / 8, nb_out = (J.n + J.shift + 7) / 8;
            for (int64_t j = i0 + threadIdx.x; j < min(i0 + kRebaseBlock, nb_out); j += kThreads) {
                const uint32_t lo = j >= 1 ? src[j - 1] : 0u, hi = j < nb_in ? src[j] : 0u;
                dst[j] = static_cast<uint8_t>((hi << J.shift) | (lo >> (8 - J.shift)));
            }
        }
    }
}

int grid_of(const Launch& L, const void* fn) {
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kThreads, 0);
    return L.sm_count * (per_sm > 0 ? per_sm : 1);
}

}  // namespace

int64_t tables_rebase_blocks(const RebaseJob& j) {
    const int64_t n = j.shift ? (j.n + j.shift + 7) / 8 : j.n;
    return (n + kRebaseBlock - 1) / kRebaseBlock;
}

void k_tables_rebase(const Launch& L, const RebaseJob* jobs, uint32_t n_jobs, int64_t n_blocks) {
    const int grid = static_cast<int>(std::min<int64_t>(n_blocks, static_cast<int64_t>(L.sm_count) * 8));
    tables_rebase_kernel<<<grid, kThreads, 0, L.stream>>>(jobs, n_jobs, n_blocks);
}

int64_t tables_tile_lines(uint32_t n_ext) {
    // keeps the count matrix (E x tiles) at <= 1 entry per 32 lines
    return n_ext <= 64 ? 2048 : static_cast<int64_t>(n_ext) * 32;
}

void k_tables_count(const Launch& L, const int32_t* ext_id, int64_t n_lines, uint32_t n_ext, int64_t tile_lines, int64_t n_tiles, uint32_t* counts) {
    const int w = tile_warps(n_ext);
    tables_count_kernel<<<static_cast<unsigned>((n_tiles + w - 1) / w), 32 * w, static_cast<size_t>(w) * n_ext * 4, L.stream>>>(
        ext_id, n_lines, n_ext, tile_lines, n_tiles, counts);
}

void k_tables_layout(const Launch& L, const int64_t* starts, int64_t n_tiles, uint32_t n_ext, const uint32_t* slots, bool with_groups,
                     TableLayout* lay) {
    tables_layout_kernel<<<1, 1024, static_cast<size_t>(n_ext) * 12, L.stream>>>(starts, n_tiles, n_ext, slots, with_groups ? 1u : 0u, lay);
}

void k_tables_scatter(const Launch& L, const int32_t* ext_id, int64_t n_lines, uint32_t n_ext, int64_t tile_lines, int64_t n_tiles,
                      const int64_t* starts, const TableLayout* lay, int64_t* rows) {
    const int w = tile_warps(n_ext);
    tables_scatter_kernel<<<static_cast<unsigned>((n_tiles + w - 1) / w), 32 * w, static_cast<size_t>(w) * n_ext * 8, L.stream>>>(
        ext_id, n_lines, n_ext, tile_lines, n_tiles, starts, lay, rows);
}

void k_tables_len(const Launch& L, const TableLayout* lay, uint32_t n_ext, const int64_t* rows, const int32_t* spans, uint32_t stride,
                  uint32_t* lens, uint32_t* valid, unsigned long long* stats) {
    const int grid = grid_of(L, reinterpret_cast<const void*>(tables_len_kernel));
    tables_len_kernel<<<grid, kThreads, 0, L.stream>>>(lay, n_ext, rows, spans, stride, lens, valid, stats);
}

void k_tables_gather(const Launch& L, const TableLayout* lay, uint32_t n_ext, const int64_t* rows, const int64_t* line_off, const int32_t* spans,
                     uint32_t stride, const void* text, int unit_bytes, const uint32_t* lens, int64_t* offs, const int64_t* col_info, uint8_t* data) {
    if (unit_bytes == 1) {
        const int grid = grid_of(L, reinterpret_cast<const void*>(tables_gather_kernel<uint8_t>));
        tables_gather_kernel<uint8_t><<<grid, kThreads, 0, L.stream>>>(lay, n_ext, rows, line_off, spans, stride, static_cast<const uint8_t*>(text),
                                                                       lens, offs, col_info, data);
    } else {
        const int grid = grid_of(L, reinterpret_cast<const void*>(tables_gather_kernel<uint16_t>));
        tables_gather_kernel<uint16_t><<<grid, kThreads, 0, L.stream>>>(lay, n_ext, rows, line_off, spans, stride, static_cast<const uint16_t*>(text),
                                                                         lens, offs, col_info, data);
    }
}

}  // namespace gorp
