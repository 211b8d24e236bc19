// Engine + C ABI of libgorpcuda (include/gorp_cuda.h). Host orchestration only; the kernels are in kernels/.
//
// Device pipeline per batch (one stream, no host round trip except reading the line count of the text form):
//   text form            : K1 count -> scan -> K1 scatter -> K1 finish          => line_off[n+1], n_lines
//                          (the List<String> form brings its own line index: the caller's offsets)
//   small definitions    : fused walk (kernels/tailwalk.cu, "all" mode) over the line index => ext_id, spans, histogram
//   big definitions      : K2b line walk over the early-exit table => candidates -> K3 histogram -> bucket pass ->
//                          K4c tail walk (+ K4b capture walk for extractions without a tail) => ext_id, spans
//   fallbacks            : K2 dfa_scan, K4 tdfa_capture (one line per thread)
#include <cuda_runtime.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/gorp_cuda.h"
#include "host/fused.hpp"
#include "host/walktables.hpp"
#include "kernels/kernels.cuh"

using namespace gorp;

namespace {

thread_local std::string g_error;

int fail(int code, const std::string& msg) {
    g_error = msg;
    return code;
}

struct CudaError : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct ArgError : std::runtime_error {  // bad input data (reported as GORP_E_ARG)
    using std::runtime_error::runtime_error;
};

#define CK(expr)                                                                                                   \
    do {                                                                                                           \
        cudaError_t _e = (expr);                                                                                   \
        if (_e != cudaSuccess)                                                                                     \
            throw CudaError(std::string(#expr) + ": " + cudaGetErrorName(_e) + " (" + cudaGetErrorString(_e) + ")"); \
    } while (0)

template <class F>
int guarded(F&& f) {
    try {
        return f();
    } catch (const DefinitionParseError& e) {
        return fail(GORP_E_DEFINITION, e.what());
    } catch (const UnsupportedError& e) {
        return fail(GORP_E_UNSUPPORTED, e.what());
    } catch (const BlobError& e) {
        return fail(GORP_E_BLOB, e.what());
    } catch (const CudaError& e) {
        return fail(GORP_E_CUDA, e.what());
    } catch (const ArgError& e) {
        return fail(GORP_E_ARG, e.what());
    } catch (const std::bad_alloc&) {
        return fail(GORP_E_OOM, "out of host memory");
    } catch (const std::exception& e) {
        return fail(GORP_E_INTERNAL, e.what());
    }
}

// ------------------------------------------------------------------ device buffers
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        if (p) CK(cudaFree(p));
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            want = bytes;
            CK(cudaMalloc(&p, want));
        }
        cap = want;
    }
    // grows to at least `bytes`, keeping the first `keep` bytes (device-to-device copy on `stream`, then waits)
    void grow_keep(size_t bytes, size_t keep, cudaStream_t stream) {
        if (bytes <= cap) return;
        DevBuf bigger;
        bigger.reserve(bytes);
        if (p && keep) {
            CK(cudaMemcpyAsync(bigger.p, p, keep, cudaMemcpyDeviceToDevice, stream));
            CK(cudaStreamSynchronize(stream));
        }
        std::swap(p, bigger.p);
        std::swap(cap, bigger.cap);
    }
    template <class T>
    T* as() const { return static_cast<T*>(p); }
    ~DevBuf() {
        if (p) cudaFree(p);
    }
};

template <class T>
T* upload(const std::vector<T>& v, std::vector<void*>& owned) {
    void* p = nullptr;
    CK(cudaMalloc(&p, std::max<size_t>(v.size() * sizeof(T), 16)));
    owned.push_back(p);
    if (!v.empty()) CK(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return static_cast<T*>(p);
}

// The host descriptors of a gorp_device_tables: one gorp_value_table per extraction, and per column (of all tables, in
// table order) the pointers and null count the tables point into.
struct TableDescs {
    std::vector<gorp_value_table> tables;
    std::vector<const int64_t*> offsets;
    std::vector<const void*> data;
    std::vector<const uint8_t*> valid;
    std::vector<int64_t> nulls;
    void reset(size_t n_tables, int64_t n_cols) {
        tables.assign(n_tables, gorp_value_table{});
        offsets.assign(static_cast<size_t>(n_cols), nullptr);
        data.assign(static_cast<size_t>(n_cols), nullptr);
        valid.assign(static_cast<size_t>(n_cols), nullptr);
        nulls.assign(static_cast<size_t>(n_cols), 0);
    }
    // table t: columns [col_base, col_base + n_cols) of the column arrays
    void set_table(size_t t, int64_t n_rows, const int64_t* rows, int64_t col_base, int64_t n_cols) {
        gorp_value_table& v = tables[t];
        v.n_rows = n_rows;
        v.n_columns = static_cast<int32_t>(n_cols);
        v.d_row = rows;
        if (n_cols) {
            v.d_offsets = offsets.data() + col_base;
            v.d_data = data.data() + col_base;
            v.d_valid = valid.data() + col_base;
            v.null_count = nulls.data() + col_base;
        }
    }
    void describe(gorp_device_tables* out, int unit_bytes) const {
        out->n_tables = static_cast<int32_t>(tables.size());
        out->unit_bytes = unit_bytes;
        out->tables = tables.data();
    }
};

constexpr int kMaxTimed = 16;
struct DeviceCtx {
    int device = 0;
    int numa_node = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    std::vector<void*> owned;  // immutable tables
    DfaDev dfa{};
    DfaDirectDev dfa_direct{};
    TdfaFastDev cap_fast{};
    CapDev cap{};
    DfaWalkDev dfawalk{};        // class-indexed combined DFA of kernels/dfawalk.cu (text form, any definition)
    PikeDev pike{};              // simulating Pike VM for extractions without a determinised capture automaton (kernels/pike.cu)
    DevBuf pike_scratch;
    MatchAllDev matchall{};      // the reference's own tables (matchAll)
    DevBuf ma_state, ma_count, ma_off, ma_out;
    DfaWalkDev dfawalk_cut{};    // the same with the early-exit cut of host/tails.hpp (K2b when the tail walk follows)
    TailDev tails{};             // per-extraction tail automata of kernels/tailwalk.cu
    TailDev fused_tail{};        // the one-pass automaton of host/fused.hpp as ONE tail table for every line (K1 + tail walk, "fused walk")
    uint32_t tail_flush_every = 8;  // walk iterations per round of the tail walk (GORP_TAIL_FLUSH)
    uint32_t item_lines = kCapItemLines;  // work items of the capture walks (GORP_ITEM_LINES)
    bool item_interleave = false;         // ... listed by relative position inside their bucket (GORP_ITEM_ORDER=1)
    DevBuf long_lines, recs;
    CapImgDev capimg{};          // per-extraction capture tables of kernels/capwalk.cu (text form, any definition)
    bool force_k4 = false;       // GORP_FORCE_K4=1: one-line-per-thread capture kernels (K4) instead of the bucketed K4b
    DevBuf perm, items, buckets, nl_masks;
    bool force_k1k2 = false;     // GORP_FORCE_K1K2=1: newline index without masks + one-line-per-thread DFA scan (K1, K2) instead of K2b
    uint32_t* d_slots = nullptr;
    uint32_t n_ext = 0;
    uint32_t max_slots = 0;
    bool force_general = false;  // GORP_FORCE_GENERAL=1: always use the general (masked) kernels
    bool force_twopass = false;  // GORP_FORCE_TWOPASS=1: never use the fused walk (small definitions take the big-definition path)
    double lines_per_unit = 1.0 / 24.0;  // running estimate that sizes the row arrays of a host-buffer call (run_pieces)
    // host-buffer calls are pipelined in pieces: H2D of piece k+1 (s_in) overlaps the kernels of piece k (stream) and
    // the D2H of the rows of piece k-1 (s_out); the rows of all pieces accumulate in acc_*
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2]{}, ev_free[2]{}, ev_rows = nullptr;
    cudaEvent_t ev_done = nullptr;  // end of the last call on this context: the next call's stream waits for it (shared scratch)
    DevBuf textbuf[2], offbuf[2], bytebuf[2], acc_ext, acc_off, acc_spans, acc_hist;
    DevBuf byte_off;  // byte line offsets of a UTF-8 piece (byte coordinates)
    DevBuf unit_off, slice_units;  // UTF-8 strings (gorp_extract_lines_utf8): unit offsets of the piece's strings, count-pass slice prefixes
    // per-call scratch, serialised by `mu`
    std::mutex mu;
    DevBuf text, off_in, line_off, tile_counts, tile_base, scan_scratch, ext_id, spans, hist, scalars;
    // the result of the last successful device-resident extract call, which gorp_extract_tables_device reads; every other
    // call that takes `mu` through CtxLock forgets it (its scratch may hold something else by then)
    int last_unit_bytes = 0;  // 2: a UTF-16 call, 1: a UTF-8 call, 0: none
    const void* last_text = nullptr;
    gorp_device_result last{};
    // value tables of gorp_extract_tables_device: device buffers, and the host descriptors the caller reads
    DevBuf tb_counts, tb_starts, tb_scan, tb_layout, tb_rows, tb_lens, tb_valid, tb_stats, tb_offs, tb_colinfo, tb_data;
    TableDescs tb_desc;
    // tables of the UTF-8 host calls: the device's whole byte range [R0, R1) of the batch, the merge jobs and the shifted
    // bitmaps of a call on several devices
    DevBuf resident, tb_jobs, tb_stage;
    // per-kernel device time: CUDA events on the launching stream, accumulated over timed calls
    cudaEvent_t ev[kMaxTimed + 1]{};
    const char* ev_name[kMaxTimed]{};
    int n_ev = 0;             // events pending collection (recorded by the last timed call)
    double acc_ms[kMaxTimed]{};
    int64_t acc_calls = 0;
    int acc_n = 0;
    int64_t launches = 0;     // kernels launched by this context (all calls)

    ~DeviceCtx() {
        cudaSetDevice(device);
        for (void* p : owned) cudaFree(p);
        for (auto& e : ev)
            if (e) cudaEventDestroy(e);
        for (auto& e : ev_in)
            if (e) cudaEventDestroy(e);
        for (auto& e : ev_free)
            if (e) cudaEventDestroy(e);
        if (ev_rows) cudaEventDestroy(ev_rows);
        if (ev_done) cudaEventDestroy(ev_done);
        if (stream) cudaStreamDestroy(stream);
        if (s_in) cudaStreamDestroy(s_in);
        if (s_out) cudaStreamDestroy(s_out);
    }
};

// Holds c.mu for an extract or match call: the device-resident result that gorp_extract_tables_device reads does not
// survive it (a device-resident call that succeeds records its own result again).
struct CtxLock {
    std::unique_lock<std::mutex> lock;
    explicit CtxLock(DeviceCtx& c) : lock(c.mu) { c.last_unit_bytes = 0; }
};

// NUMA node of a CUDA device (sysfs numa_node of its PCI function), or -1 when the platform does not say
int device_numa_node(int device) {
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), device) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    for (char* p = bdf; *p; ++p) *p = static_cast<char>(std::tolower(*p));
    const std::string path = std::string("/sys/bus/pci/devices/") + bdf + "/numa_node";
    FILE* f = std::fopen(path.c_str(), "r");
    if (!f) return -1;
    int node = -1;
    if (std::fscanf(f, "%d", &node) != 1) node = -1;
    std::fclose(f);
    return node;
}

// While alive, the calling thread prefers `node` for new pages (set_mempolicy MPOL_PREFERRED): pinned result / staging
// buffers are allocated next to the GPU that fills them, so the D2H copies of several GPUs do not all cross the socket
// interconnect. A no-op where the node is unknown or the syscall is not permitted.
struct NumaPrefer {
    bool set = false;
    explicit NumaPrefer(int node) {
#ifdef SYS_set_mempolicy
        if (node < 0 || node >= 1024) return;
        unsigned long mask[16] = {0};
        mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
        set = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, sizeof(mask) * 8 + 1) == 0;
#else
        (void)node;
#endif
    }
    ~NumaPrefer() {
#ifdef SYS_set_mempolicy
        if (set) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0);
#endif
    }
};

// Pinned host arrays behind a gorp_result: 0-3 ext_id, line_off, spans, histogram; with value tables (the *_tables calls)
// 4-7 row indexes, offsets, values and bitmaps of every table, described by `tables`.
struct HostResult {
    int numa_node = -1;  // of the device that fills the arrays (first device of the engine)
    void* p[8] = {};
    size_t cap[8] = {};
    TableDescs tables;
    void reserve(int i, size_t bytes, size_t keep = 0) {  // keeps the first `keep` bytes when it has to grow
        if (bytes <= cap[i]) return;
        void* q = nullptr;
        size_t want = bytes + bytes / 8 + 64;
        {
            NumaPrefer near_the_gpu(numa_node);
            CK(cudaMallocHost(&q, want));
        }
        if (p[i] && keep) std::memcpy(q, p[i], keep);
        if (p[i]) cudaFreeHost(p[i]);
        p[i] = q;
        cap[i] = want;
    }
    ~HostResult() {
        for (auto q : p)
            if (q) cudaFreeHost(q);
    }
};

}  // namespace

struct gorp_engine {
    CompiledDefinition def;
    bool match_only = false;
    std::vector<std::unique_ptr<DeviceCtx>> devs;
    std::mutex pool_mu;
    std::vector<std::unique_ptr<HostResult>> pool;
};

namespace {

// Uploads a tail image (host/walktables.hpp) and fills the device descriptor of kernels/tailwalk.cu.
void upload_tail_image(const TailImage& img, const TailSet& T, uint32_t span_stride, TailDev& d, std::vector<void*>& owned) {
    static_assert(sizeof(TailImageExt) == sizeof(TailExt), "host and device descriptors of a tail table must match");
    std::vector<TailExt> text(img.ext.size());
    std::memcpy(text.data(), img.ext.data(), text.size() * sizeof(TailExt));
    d.image = upload(img.image, owned);
    d.ext = upload(text, owned);
    d.res = upload(img.res, owned);
    d.oext = upload(img.oext, owned);
    d.init_slots = upload(img.init_slots, owned);
    d.xcol = upload(T.xcol, owned);
    d.pair_col = upload(T.pair_col, owned);
    d.width = img.width;
    d.row_bytes = img.row_bytes;
    d.span_stride = span_stride;
    d.max_table_bytes = img.max_table_bytes;
    d.max_slots = img.max_slots;
    d.nl_data_col = T.nl_data_col;
    for (const TailImageExt& x : img.ext) {
        if (!x.available) {
            ++d.n_without;
            continue;
        }
        d.max_res = std::max(d.max_res, (x.n_outcomes * span_stride + 3u) & ~3u);
        d.max_outcomes = std::max(d.max_outcomes, (x.n_outcomes + 3u) & ~3u);
    }
}

void build_device(DeviceCtx& c, const DeviceModel& m, const FusedAutomaton& fused, const TailSet& tailset, const DfaTables& raw,
                  bool match_only) {
    CK(cudaSetDevice(c.device));
    cudaDeviceProp prop{};
    CK(cudaGetDeviceProperties(&prop, c.device));
    c.sm_count = prop.multiProcessorCount;
    c.numa_node = device_numa_node(c.device);
    CK(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c.s_in, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c.s_out, cudaStreamNonBlocking));
    for (auto& e : c.ev_in) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto& e : c.ev_free) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c.ev_rows, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c.ev_done, cudaEventDisableTiming));
    if (const char* f = std::getenv("GORP_FORCE_GENERAL")) c.force_general = f[0] == '1';
    if (const char* f = std::getenv("GORP_FORCE_TWOPASS")) c.force_twopass = f[0] == '1';
    if (const char* f = std::getenv("GORP_FORCE_K1K2")) c.force_k1k2 = f[0] == '1';
    if (const char* f = std::getenv("GORP_FORCE_K4")) c.force_k4 = f[0] == '1';
    if (const char* f = std::getenv("GORP_L2_FETCH")) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, static_cast<size_t>(std::atoi(f)));  // diagnostics
    for (auto& e : c.ev) CK(cudaEventCreate(&e));
    // the reference's tables as they are (matchAll)
    c.matchall.classmap = upload(raw.classmap, c.owned);
    c.matchall.trans = upload(raw.trans, c.owned);
    c.matchall.accept_off = upload(raw.accept_off, c.owned);
    c.matchall.accept_list = upload(raw.accept_list, c.owned);
    c.matchall.n_classes = raw.n_classes;
    // combined DFA
    const size_t S = m.dfa.n_states, C = m.dfa.n_classes;
    c.dfa.n_states = static_cast<uint32_t>(S);
    c.dfa.n_classes = static_cast<uint32_t>(C);
    c.dfa.cls = upload(m.dfa.classmap, c.owned);
    {
        // device layout: one extra absorbing "dead" row and one extra "identity" column (see kernels.cu)
        const size_t R = S + 1, K = C + 1;
        std::vector<int32_t> af(m.dfa.accept_first);
        af.push_back(-1);
        c.dfa.accept_first = upload(af, c.owned);
        if (R * K > 0x7FFFFFFFull) throw UnsupportedError("combined DFA table too large");
        auto next = [&](size_t s, size_t k) -> uint32_t {
            if (s == S) return static_cast<uint32_t>(S * K);
            if (k == C) return static_cast<uint32_t>(s * K);
            int32_t t = m.dfa.trans[s * C + k];
            return static_cast<uint32_t>((t < 0 ? S : static_cast<size_t>(t)) * K);
        };
        if (R * K <= 0xFFFF) {
            std::vector<uint16_t> t(R * K);
            for (size_t s = 0; s < R; ++s)
                for (size_t k = 0; k < K; ++k) t[s * K + k] = static_cast<uint16_t>(next(s, k));
            c.dfa.trans = upload(t, c.owned);
            c.dfa.wide = 0;
        } else {
            std::vector<uint32_t> t(R * K);
            for (size_t s = 0; s < R; ++s)
                for (size_t k = 0; k < K; ++k) t[s * K + k] = next(s, k);
            c.dfa.trans = upload(t, c.owned);
            c.dfa.wide = 1;
        }
    }
    // fast tier: directly ASCII-indexed rows (see kernels.cuh: DfaDirectDev)
    {
        const size_t E = m.n_groups.size();
        const size_t skip_base = S, fin_base = S + 7, R = fin_base + 1 + E;
        if (R * 512 <= 96 * 1024) {
            std::vector<uint32_t> rows(R * 128);
            for (size_t r = 0; r < R; ++r)
                for (size_t u = 0; u < 128; ++u) {
                    uint32_t nx;
                    if (r < S) {
                        if (u == 0x0A) {
                            nx = static_cast<uint32_t>(fin_base + 1 + m.dfa.accept_first[r]);
                        } else {
                            int32_t t = m.dfa.trans[r * C + m.dfa.classmap[u]];
                            nx = t < 0 ? static_cast<uint32_t>(fin_base) : static_cast<uint32_t>(t);
                        }
                    } else if (r < fin_base) {
                        nx = r == skip_base ? 0u : static_cast<uint32_t>(r - 1);
                    } else {
                        nx = static_cast<uint32_t>(r);
                    }
                    rows[r * 128 + u] = nx;
                }
            c.dfa_direct.rows = upload(rows, c.owned);
            c.dfa_direct.n_rows = static_cast<uint32_t>(R);
            c.dfa_direct.n_states = static_cast<uint32_t>(S);
            c.dfa_direct.skip_base = static_cast<uint32_t>(skip_base);
            c.dfa_direct.fin_base = static_cast<uint32_t>(fin_base);
            c.dfa_direct.cls = c.dfa.cls;
            c.dfa_direct.trans_plain = upload(m.dfa.trans, c.owned);
            c.dfa_direct.accept_first = c.dfa.accept_first;
            c.dfa_direct.n_classes = static_cast<uint32_t>(C);
            c.dfa_direct.enabled = 1;
        }
    }
    // line-walk DFA tier (K2b): class-indexed u16 rows + DEADSCAN / SKIP / FIN rows (host/walktables.hpp)
    if (!std::getenv("GORP_SKIP_NEWTABLES")) {
        const DfaWalkTable t = build_dfawalk_table(m);
        if (t.available) {
            c.dfawalk.table = upload(t.rows, c.owned);
            c.dfawalk.n_rows = t.n_rows;
            c.dfawalk.K = t.K;
            c.dfawalk.n_states = t.n_states;
            c.dfawalk.fin_base = t.fin_base;
            c.dfawalk.cls128 = upload(t.cls128, c.owned);
            c.dfawalk.xcls = upload(t.xcls, c.owned);
            c.dfawalk.enabled = 1;
        }
    }
    // capture automata
    const size_t E = m.n_groups.size();
    c.n_ext = static_cast<uint32_t>(E);
    std::vector<uint32_t> slots(E);
    for (size_t e = 0; e < E; ++e) slots[e] = 2 * m.n_groups[e];
    c.d_slots = upload(slots, c.owned);
    for (uint32_t v : slots) c.max_slots = std::max(c.max_slots, v);
    c.cap.n_ext = static_cast<uint32_t>(E);
    c.cap.match_only = match_only ? 1u : 0u;
    if (!match_only) {
        std::vector<ExtDev> ext(E);
        std::vector<uint32_t> trans, opoff;
        std::vector<uint16_t> ops;
        std::vector<uint8_t> fin, acc;
        for (size_t e = 0; e < E; ++e) {
            const Tdfa& t = m.tdfas[e];
            if (t.n_regs > static_cast<uint32_t>(kMaxTdfaRegsBig))
                throw UnsupportedError(strfmt("extraction #%zu needs %u tag registers (limit %d)", e, t.n_regs, kMaxTdfaRegsBig));
            c.cap.max_regs = std::max(c.cap.max_regs, t.n_regs);
            ext[e] = {t.n_states, static_cast<uint32_t>(trans.size()), static_cast<uint32_t>(opoff.size()),
                      static_cast<uint32_t>(ops.size()), static_cast<uint32_t>(fin.size()), static_cast<uint32_t>(acc.size()),
                      t.n_slots};
            // rows + dead row, columns + identity column
            const uint32_t Sd = t.n_states, Cn = t.n_classes;
            for (uint32_t s = 0; s <= Sd; ++s) {
                for (uint32_t k = 0; k < Cn; ++k) {
                    uint32_t ent = s == Sd ? 0xFFFFu : t.trans[static_cast<size_t>(s) * Cn + k];
                    if ((ent & 0xFFFFu) == 0xFFFFu) ent = Sd;  // dead: no register ops
                    trans.push_back(ent);
                }
                trans.push_back(s);  // identity: stay, no ops
            }
            opoff.insert(opoff.end(), t.op_off.begin(), t.op_off.end());
            ops.insert(ops.end(), t.ops.begin(), t.ops.end());
            fin.insert(fin.end(), t.fin.begin(), t.fin.end());
            fin.insert(fin.end(), t.n_slots, 0xFF);
            acc.insert(acc.end(), t.accepting.begin(), t.accepting.end());
            acc.push_back(0);
        }
        // fast tier image: cls128 (class*4, '\n' -> dedicated column) + per-extraction tables (kernels.cuh: TdfaFastDev)
        {
            const uint32_t Cn = m.symbols.n_classes, K = Cn + 1, NL = Cn, row_bytes = K * 4;
            std::vector<uint32_t> image(128);
            for (uint32_t u = 0; u < 128; ++u) image[u] = (u == 0x0A ? NL : m.symbols.classmap[u]) * 4;
            std::vector<FastExtDev> fext(E);
            uint32_t max_regs = 0;
            bool ok = true;
            for (size_t e = 0; e < E && ok; ++e) {
                const Tdfa& t = m.tdfas[e];
                const uint32_t Sx = t.n_states, rows = 2 * Sx + 9;
                if (static_cast<uint64_t>(rows) * row_bytes > 0xFFFC) { ok = false; break; }
                max_regs = std::max(max_regs, t.n_regs);
                fext[e] = {static_cast<uint32_t>(image.size() * 4), row_bytes, Sx, (Sx + 7) * row_bytes, (Sx + 8) * row_bytes,
                           (Sx + 9) * row_bytes};
                const size_t base = image.size();
                image.resize(base + static_cast<size_t>(rows) * K);
                auto put = [&](uint32_t r, uint32_t k, uint32_t next_row, uint32_t dst) {
                    image[base + static_cast<size_t>(r) * K + k] = (next_row * row_bytes) | (dst << 16);
                };
                for (uint32_t r = 0; r < rows; ++r)
                    for (uint32_t k = 0; k < K; ++k) {
                        if (r < Sx) {
                            if (k == NL) { put(r, k, Sx + 9 + r, 0xFFFE); continue; }  // LEN := position of the '\n'
                            const uint32_t ent = t.trans[static_cast<size_t>(r) * Cn + k];
                            const uint32_t nx = ent & 0xFFFFu, ol = ent >> 16;
                            if (nx == 0xFFFFu) { put(r, k, Sx + 7, 0xFFFF); continue; }
                            const uint32_t o0 = t.op_off[ol], o1 = t.op_off[ol + 1];
                            if (o1 == o0) put(r, k, nx, 0xFFFF);
                            else if (o1 - o0 == 1 && (t.ops[o0] & 0xFF) == 0xFF) put(r, k, nx, t.ops[o0] >> 8);
                            else put(r, k, Sx + 8, 0xFFFF);  // SLOW: replayed through the general tables
                        } else if (r < Sx + 7) {
                            put(r, k, r == Sx ? 0u : r - 1, 0xFFFF);  // SKIP chain
                        } else {
                            put(r, k, r, 0xFFFF);  // DEAD / SLOW / FRZ: absorbing
                        }
                    }
            }
            while (image.size() % 4) image.push_back(0);  // keep what follows the image 16-byte aligned in shared memory
            const uint32_t reg_stride = kCapFastThreads * 4;
            const size_t reg_bytes = static_cast<size_t>(max_regs + 2) * reg_stride;
            if (ok && image.size() * 4 + reg_bytes <= 160 * 1024 && (max_regs + 2) * reg_stride <= 0x10000) {
                // resolve the register byte offsets now that the register count is known:
                // r -> r*stride, dummy -> max_regs*stride, LEN -> (max_regs+1)*stride
                for (size_t i = 128; i < image.size(); ++i) {
                    uint32_t dst = image[i] >> 16;
                    dst = dst == 0xFFFF ? max_regs : (dst == 0xFFFE ? max_regs + 1 : dst);
                    image[i] = (image[i] & 0xFFFFu) | ((dst * reg_stride) << 16);
                }
                c.cap_fast.image = upload(image, c.owned);
                c.cap_fast.image_words = static_cast<uint32_t>(image.size());
                c.cap_fast.n_regs = max_regs;
                c.cap_fast.ext = upload(fext, c.owned);
                c.cap_fast.enabled = 1;
            }
        }
        // bucketed capture tier: one table per extraction (host/walktables.hpp, kernels.cuh: CapImgDev)
        if (!std::getenv("GORP_SKIP_NEWTABLES")) {
            const CapImage img = build_cap_image(m, kCapMaxBuckets);
            if (img.available) {
                static_assert(sizeof(CapImageExt) == sizeof(CapImgExt), "host and device descriptors of a capture table must match");
                std::vector<CapImgExt> fext(img.ext.size());
                std::memcpy(fext.data(), img.ext.data(), fext.size() * sizeof(CapImgExt));
                c.capimg.image = upload(img.image, c.owned);
                c.capimg.cls128 = upload(img.cls128, c.owned);
                c.capimg.ext = upload(fext, c.owned);
                c.capimg.n_regs = img.n_regs;
                // shared memory for the table of the extraction a CTA works on: the largest table that still leaves room
                // for two CTAs per SM (larger tables are read through L1/L2)
                const size_t fixed = 512 + static_cast<size_t>(img.n_regs + 1) * kCapWalkThreads * 4;
                const size_t budget = fixed + 5 * 1024 < 110 * 1024 ? 110 * 1024 - fixed - 5 * 1024 : 0;
                size_t best = 0;
                for (const CapImageExt& x : img.ext)
                    if (x.frz_off <= budget) best = std::max<size_t>(best, x.frz_off);  // (S + 17) rows: without the FRZ rows
                c.capimg.smem_table_bytes = static_cast<uint32_t>((best + 15) & ~size_t(15));
                c.capimg.enabled = capwalk_smem_bytes(c.capimg) <= 200 * 1024 ? 1u : 0u;
            }
        }
        // tail tier: early-exit combined DFA + one tail automaton per extraction (host/tails.hpp, kernels/tailwalk.cu)
        if (tailset.any && c.dfawalk.enabled && c.capimg.enabled && !std::getenv("GORP_NO_TAILS")) {
            const DfaWalkTable t = build_dfawalk_table_cut(m, tailset.cut_of_state);
            const TailImage img = build_tail_image(tailset, c.max_slots);
            if (t.available && img.available) {
                TailDev& d = c.tails;
                upload_tail_image(img, tailset, c.max_slots, d, c.owned);
                if (tailwalk_smem_bytes(d, 256) <= 200 * 1024) {
                    c.dfawalk_cut.table = upload(t.rows, c.owned);
                    c.dfawalk_cut.n_rows = t.n_rows;
                    c.dfawalk_cut.K = t.K;
                    c.dfawalk_cut.n_states = t.n_states;
                    c.dfawalk_cut.fin_base = t.fin_base;
                    c.dfawalk_cut.cls128 = upload(t.cls128, c.owned);
                    c.dfawalk_cut.xcls = upload(t.xcls, c.owned);
                    c.dfawalk_cut.enabled = 1;
                    d.enabled = 1;
                    if (const char* f = std::getenv("GORP_TAIL_FLUSH")) c.tail_flush_every = std::min(64, std::max(1, std::atoi(f)));
                }
            }
        }
        // fused walk: the one-pass automaton of host/fused.hpp (DFA x capture automata folded into one automaton) laid out as ONE
        // tail table (host/tails.hpp format) that every line walks, behind the newline index K1 — lanes claim consecutive lines
        // (kernels/tailwalk.cu, `all` mode): no bucket pass
        if (fused.available && !std::getenv("GORP_NO_FUSEDWALK")) {
            const TailSet FT = build_fused_tailset(fused, m, c.max_slots);
            const TailImage img = build_tail_image(FT, c.max_slots);
            if (img.available && img.ext[0].available && c.max_slots > 0) {
                upload_tail_image(img, FT, c.max_slots, c.fused_tail, c.owned);
                c.fused_tail.enabled = tailwalk_smem_bytes(c.fused_tail, 256) <= 200 * 1024 ? 1u : 0u;
            }
        }
        c.cap.cls = upload(m.symbols.classmap, c.owned);
        c.cap.n_classes = m.symbols.n_classes;
        c.cap.pair_hi_class = m.symbols.pair_hi_class;
        c.cap.ext = upload(ext, c.owned);
        c.cap.tdfa_trans = upload(trans, c.owned);
        c.cap.tdfa_op_off = upload(opoff, c.owned);
        c.cap.tdfa_ops = upload(ops, c.owned);
        c.cap.tdfa_fin = upload(fin, c.owned);
        c.cap.tdfa_accepting = upload(acc, c.owned);
        // extractions that fall back to the simulated Pike VM
        bool any_pike = false;
        for (uint8_t v : m.pike_only) any_pike = any_pike || v;
        if (any_pike) {
            std::vector<PikeExtDev> px(E, PikeExtDev{});
            std::vector<uint32_t> clo_off;
            std::vector<int32_t> clo_target;
            std::vector<unsigned long long> clo_mask;
            std::vector<uint8_t> accepts;
            for (size_t e = 0; e < E; ++e) {
                if (!m.pike_only[e]) continue;
                const PikeTables& t = m.pike[e];
                px[e] = {static_cast<uint32_t>(clo_off.size()), t.n_insts, t.n_slots, static_cast<uint32_t>(accepts.size()), 1u};
                const uint32_t base = static_cast<uint32_t>(clo_target.size());
                for (uint32_t v : t.clo_off) clo_off.push_back(base + v);
                clo_target.insert(clo_target.end(), t.clo_target.begin(), t.clo_target.end());
                for (uint64_t v : t.clo_mask) clo_mask.push_back(v);
                accepts.insert(accepts.end(), t.accepts.begin(), t.accepts.end());
                c.pike.max_insts = std::max(c.pike.max_insts, t.n_insts);
                c.pike.max_slots = std::max(c.pike.max_slots, t.n_slots);
            }
            c.pike.ext = upload(px, c.owned);
            c.pike.clo_off = upload(clo_off, c.owned);
            c.pike.clo_target = upload(clo_target, c.owned);
            c.pike.clo_mask = upload(clo_mask, c.owned);
            c.pike.accepts = upload(accepts, c.owned);
            c.pike.cls = c.cap.cls;
            c.pike.n_classes = m.symbols.n_classes;
            c.pike.pair_hi_class = m.symbols.pair_hi_class;
            c.pike.enabled = 1;
        }
    }
}

void collect_times(DeviceCtx& c) {
    if (c.n_ev == 0) return;
    cudaEventSynchronize(c.ev[c.n_ev]);
    for (int i = 0; i < c.n_ev; ++i) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, c.ev[i], c.ev[i + 1]);
        c.acc_ms[i] += ms;
    }
    c.acc_n = c.n_ev;
    c.acc_calls += 1;
    c.n_ev = 0;
}

// restores the calling thread's current CUDA device when a call returns
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() {
        if (cudaGetDevice(&prev) != cudaSuccess) {
            cudaGetLastError();
            prev = -1;
        }
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

struct Timer {
    DeviceCtx& c;
    cudaStream_t s;
    bool on;
    Timer(DeviceCtx& c_, cudaStream_t s_, bool on_) : c(c_), s(s_), on(on_) {
        if (on) {
            collect_times(c);  // the previous timed call, if any
            cudaEventRecord(c.ev[0], s);
        }
    }
    void mark(const char* name, int launches) {
        c.launches += launches;
        if (!on || c.n_ev >= kMaxTimed) return;
        c.ev_name[c.n_ev] = name;
        ++c.n_ev;
        cudaEventRecord(c.ev[c.n_ev], s);
    }
};

// Runs the device pipeline. Text form when d_off == nullptr. Caller holds c.mu and has set the device; `tm` times the
// stages of the caller's call on `stream`.
// Returns n_lines (synchronises once for the text form to size the per-line arrays).
int64_t run_pipeline_tables(DeviceCtx& c, const uint16_t* d_text, int64_t n_units, const int64_t* d_off, int64_t n_lines,
                            cudaStream_t stream, Timer& tm, gorp_device_result* out);

// The table-driven pipeline, then (only for definitions that have such extractions) the simulated Pike VM over the lines
// that came out as CAPTURE_FAIL of an extraction without a determinised capture automaton.
int64_t run_pipeline(DeviceCtx& c, const uint16_t* d_text, int64_t n_units, const int64_t* d_off, int64_t n_lines,
                     cudaStream_t stream, Timer& tm, gorp_device_result* out) {
    gorp_device_result local{};
    gorp_device_result* r = out ? out : &local;
    const int64_t nl = run_pipeline_tables(c, d_text, n_units, d_off, n_lines, stream, tm, r);
    if (c.pike.enabled && nl > 0 && !c.cap.match_only) {
        Launch L{stream, c.sm_count};
        const size_t per_thread = pike_scratch_ints_per_thread(c.pike) * 4;
        size_t threads = static_cast<size_t>(c.sm_count) * 128;
        const size_t budget = 256ull << 20;
        if (threads * per_thread > budget) threads = std::max<size_t>(128, budget / per_thread / 128 * 128);
        c.pike_scratch.reserve(threads * per_thread);
        // (the result arrays are the engine's own buffers: const only in the caller's view)
        k_pike_fixup(L, c.pike, d_text, r->d_line_off, d_off ? 0 : 1, nl, c.max_slots, const_cast<int32_t*>(r->d_ext_id),
                     const_cast<int32_t*>(r->d_spans), reinterpret_cast<unsigned long long*>(const_cast<int64_t*>(r->d_histogram)), c.n_ext,
                     c.pike_scratch.as<int32_t>(), static_cast<uint32_t>(threads));
        tm.mark("pike_fixup", 1);
        CK(cudaGetLastError());
    }
    return nl;
}

int64_t run_pipeline_tables(DeviceCtx& c, const uint16_t* d_text, int64_t n_units, const int64_t* d_off, int64_t n_lines,
                            cudaStream_t stream, Timer& tm, gorp_device_result* out) {
    Launch L{stream, c.sm_count};
    c.scalars.reserve(128);
    int64_t* d_n_lines = c.scalars.as<int64_t>();
    const int64_t* d_line_off;
    int sep;
    bool ends_with_nl = true;
    if (!d_off) {  // text form: the newline index K1
        sep = 1;
        const int64_t n_tiles = (n_units + kNlTile - 1) / kNlTile;
        c.tile_counts.reserve(static_cast<size_t>(n_tiles + 1) * 4);
        c.tile_base.reserve(static_cast<size_t>(n_tiles + 2) * 8);
        c.scan_scratch.reserve(static_cast<size_t>(n_tiles / 4096 + 8) * 8);
        const bool with_masks = !c.force_k1k2 && !c.force_general;  // the count pass leaves the '\n' masks for the scatter pass
        if (with_masks) {
            c.nl_masks.reserve(static_cast<size_t>(n_tiles + 4) * 256 * 4);
            k1_count_newlines_masks(L, d_text, n_units, c.tile_counts.as<uint32_t>(), c.nl_masks.as<uint32_t>());
        } else {
            k1_count_newlines(L, d_text, n_units, c.tile_counts.as<uint32_t>());
        }
        tm.mark("k1_count_newlines", 1);
        scan_u32_to_i64(L, c.tile_counts.as<uint32_t>(), n_tiles, c.tile_base.as<int64_t>(), c.scan_scratch.as<int64_t>());
        tm.mark("scan_tiles", 3);
        // the one host round trip of the text form: the newline total (and the last unit) size the per-line arrays
        int64_t total_nl = 0;
        uint16_t last_unit = 0x0A;
        CK(cudaMemcpyAsync(&total_nl, c.tile_base.as<int64_t>() + n_tiles, 8, cudaMemcpyDeviceToHost, stream));
        if (n_units > 0) CK(cudaMemcpyAsync(&last_unit, d_text + n_units - 1, 2, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        n_lines = total_nl + (last_unit != 0x0A ? 1 : 0);
        ends_with_nl = last_unit == 0x0A;
        if (n_units > 0) c.lines_per_unit = std::max(static_cast<double>(n_lines) / static_cast<double>(n_units), 1e-6);
        c.line_off.reserve(static_cast<size_t>(total_nl + 3) * 8);
        if (with_masks) k1_scatter_masks(L, c.nl_masks.as<uint32_t>(), n_units, c.tile_base.as<int64_t>(), c.line_off.as<int64_t>());
        else k1_scatter_newlines(L, d_text, n_units, c.tile_base.as<int64_t>(), c.line_off.as<int64_t>());
        k1_finish(L, d_text, n_units, c.tile_base.as<int64_t>() + n_tiles, c.line_off.as<int64_t>(), d_n_lines);
        tm.mark("k1_scatter_newlines", 2);
        d_line_off = c.line_off.as<int64_t>();
    } else {
        sep = 0;
        d_line_off = d_off;
        CK(cudaMemcpyAsync(d_n_lines, &n_lines, 8, cudaMemcpyHostToDevice, stream));
    }
    const size_t nl = static_cast<size_t>(n_lines);
    c.ext_id.reserve((nl + 1) * 4);
    c.hist.reserve((c.n_ext + 2) * 8);
    // small definitions: the fused walk — every line through the one-pass automaton laid out as a tail table
    const bool fusedwalk = c.fused_tail.enabled && (!d_off || n_units > 0) && !c.force_twopass && !c.force_general && !c.force_k1k2 &&
                           !c.force_k4 && !c.cap.match_only && c.max_slots > 0 && (reinterpret_cast<uintptr_t>(d_text) & 31) == 0;
    if (fusedwalk && n_lines > 0 && n_lines < (1ll << 32)) {
        const uint32_t stride = c.max_slots;
        size_t rows = nl;  // GORP_PAD_ROWS (diagnostics): spare rows, which shift every allocation that follows
        if (const char* f = std::getenv("GORP_PAD_ROWS")) rows += static_cast<size_t>(std::atoll(f));
        c.ext_id.reserve((rows + 1) * 4);
        c.spans.reserve((rows * stride + 4) * 4);
        c.buckets.reserve(64);
        uint32_t* ticket = c.buckets.as<uint32_t>();  // [item ticket, n_long]
        CK(cudaMemsetAsync(ticket, 0, 8, stream));
        CK(cudaMemsetAsync(c.hist.p, 0, (c.n_ext + 2) * 8, stream));
        TailWalkParams T{};
        T.text = d_text;
        T.n_units = n_units;
        T.line_off = d_line_off;
        T.item_ticket = ticket;
        T.t = c.fused_tail;
        T.n_ext = c.n_ext;
        T.round_iters = c.tail_flush_every;
        T.lines_form = sep == 0 ? 1u : 0u;  // List<String> form: the caller's offsets are the line index
        if (const char* f = std::getenv("GORP_TAIL_FLAGS")) T.flags = static_cast<uint32_t>(std::atoi(f));
        T.ext_id = c.ext_id.as<int32_t>();
        T.spans = c.spans.as<int32_t>();
        T.hist = c.hist.as<unsigned long long>();
        T.long_cap = static_cast<uint32_t>(n_units / kTailMaxLen + 2);
        c.long_lines.reserve(static_cast<size_t>(T.long_cap) * 4);
        T.long_lines = c.long_lines.as<uint32_t>();
        T.n_long = ticket + 1;
        T.all = 1;
        T.n_lines = n_lines;
        // work items are taken by WARPS: big enough that the lanes idling at the end of an item do not matter (half a line out of
        // item_lines / 32), small enough that a small batch (a 64 MB piece of a host-buffer call) has items for every warp
        const int64_t warps = 2ll * c.sm_count * 16;
        uint32_t il = 64;
        while (il < 1024 && static_cast<int64_t>(il) * 4 * warps < n_lines) il *= 2;
        T.item_lines = il;
        k4c_tailwalk(L, T);
        tm.mark("k4c_fusedwalk", 2);
        CK(cudaGetLastError());
        if (out) {
            out->n_lines = n_lines;
            out->span_stride = static_cast<int32_t>(stride);
            out->d_ext_id = c.ext_id.as<int32_t>();
            out->d_line_off = d_line_off;
            out->d_spans = c.spans.as<int32_t>();
            out->d_histogram = c.hist.as<int64_t>();
            out->d_n_lines = d_n_lines;
        }
        return n_lines;
    }
    // every line but (possibly) the last is terminated by '\n' in the text form: fast tiers; an unterminated last line
    // goes through the general kernels
    const int64_t n_fast = ends_with_nl ? n_lines : n_lines - 1;
    uint32_t lw_threads = 0;
    bool lw_smem = false;
    // the tail walk follows: the combined-DFA walk may stop at the first state that leaves one candidate extraction.
    // Both walkers also serve the List<String> form (sep == 0: lines end where the offsets say, a '\n' is content).
    const bool with_tails = c.tails.enabled && !c.cap.match_only && c.max_slots > 0 && !c.force_general && !c.force_k4 &&
                            !c.force_k1k2 && n_lines > 0 && n_lines < (1ll << 32) && (reinterpret_cast<uintptr_t>(d_text) & 31) == 0 &&
                            (sep == 1 || n_units > 0);
    const DfaWalkDev& walk_table = with_tails ? c.dfawalk_cut : c.dfawalk;
    bool candidates = false;  // ext_id holds candidates of the cut table (K2b walked it): only the tail walk may follow
    if ((sep == 1 || with_tails) && !c.force_general && !c.force_k1k2 && (reinterpret_cast<uintptr_t>(d_text) & 31) == 0 &&
               k2b_linewalk_plan(walk_table, &lw_threads, &lw_smem)) {
        candidates = with_tails;
        LineWalkParams W{};
        W.text = d_text;
        W.n_units = n_units;
        W.line_off = d_line_off;
        W.n_lines = n_lines;
        W.a = walk_table;
        W.ext_id = c.ext_id.as<int32_t>();
        W.lines_form = sep == 0 ? 1u : 0u;
        W.item_ticket = reinterpret_cast<unsigned int*>(d_n_lines + 4);
        if (const char* f = std::getenv("GORP_WALK_FLAGS")) W.flags = static_cast<uint32_t>(std::atoi(f));
        CK(cudaMemsetAsync(W.item_ticket, 0, 4, stream));
        k2b_linewalk_scan(L, W, lw_threads, lw_smem);
        tm.mark("k2b_linewalk_scan", 1);
    } else if (sep == 1 && c.dfa_direct.enabled && !c.force_general) {
        k2_dfa_direct(L, c.dfa_direct, d_text, d_line_off, n_fast, c.ext_id.as<int32_t>());
        if (n_fast < n_lines) k2_dfa_scan(L, c.dfa, d_text, d_line_off + n_fast, sep, 1, c.ext_id.as<int32_t>() + n_fast);
        tm.mark("k2_dfa_scan", n_fast < n_lines ? 2 : 1);
    } else {
        k2_dfa_scan(L, c.dfa, d_text, d_line_off, sep, n_lines, c.ext_id.as<int32_t>());
        tm.mark("k2_dfa_scan", 1);
    }
    // result rows of `spans`: max_slots entries per line, no offsets needed
    const uint32_t stride = c.max_slots;
    c.spans.reserve((nl * stride + 4) * 4);
    bool hist_done = false;
    // K4b walks 32-byte blocks with 256-bit loads, like the walkers above: a text base that is only 16-byte aligned takes K4
    if (!c.cap.match_only && stride > 0 && (sep == 1 || with_tails) && c.capimg.enabled && !c.force_general && !c.force_k4 && n_lines > 0 &&
        n_lines < (1ll << 32) && (reinterpret_cast<uintptr_t>(d_text) & 31) == 0) {
        // K4b: histogram -> buckets by extraction -> one warp per work item (kernels/capwalk.cu)
        const uint32_t E = c.n_ext;
        CK(cudaMemsetAsync(c.hist.p, 0, (E + 2) * 8, stream));
        k3_histogram(L, c.ext_id.as<int32_t>(), n_lines, E, c.hist.as<unsigned long long>());
        tm.mark("k3_histogram", 1);
        hist_done = true;
        // work items of the two capture walks: `item_lines` entries of one bucket, listed bucket by bucket or (GORP_ITEM_ORDER=1)
        // by relative position inside the bucket, so that concurrent items cover the same stretch of text
        // measured on config #4 (200 buckets, profiles/README.md round 2): bucket by bucket, 4096 lines 6.77 ms; by relative
        // position 4096 / 2048 / 1024 / 512 lines 6.02 / 5.92 / 6.23 / 7.60 ms (DRAM read 1.99x -> 1.58x the text; below 2048 the
        // barrier and table load per item cost more than the locality brings), with 2 x 512 threads 5.78 ms. Config #3 (18
        // buckets): 6.88 -> 7.11 ms — the concurrent items of a few big buckets never share text, so only many-bucket
        // definitions get the interleaved order.
        uint32_t item_lines = E >= 64 ? 2048u : c.item_lines;
        bool interleave = E >= 64 ? true : c.item_interleave;
        if (const char* f = std::getenv("GORP_ITEM_LINES")) item_lines = static_cast<uint32_t>(std::atoi(f));
        if (const char* f = std::getenv("GORP_ITEM_ORDER")) interleave = f[0] == '1';
        if (item_lines < 32 || item_lines > kCapItemLines) item_lines = kCapItemLines;
        const size_t max_items = nl / item_lines + E + 1;
        c.perm.reserve(nl * 4 + 16);
        c.items.reserve(max_items * sizeof(CapItem));
        c.buckets.reserve((2 * static_cast<size_t>(E) + 8) * 4);
        uint32_t* bucket_base = c.buckets.as<uint32_t>();
        uint32_t* cursor = bucket_base + E + 1;
        uint32_t* n_items = cursor + E;
        uint32_t* item_ticket = n_items + 1;
        uint32_t* tail_ticket = n_items + 2;  // [tail_ticket, n_long]
        const bool tails = with_tails;
        if (candidates && !tails) throw std::logic_error("early-exit candidates without the tail walk");
        if (tails) {
            CK(cudaMemsetAsync(tail_ticket, 0, 8, stream));
            c.recs.reserve(nl * sizeof(LineRec) + 16);
        }
        k4b_bucket(L, c.ext_id.as<int32_t>(), n_lines, E, c.hist.as<unsigned long long>(), bucket_base, cursor, c.perm.as<uint32_t>(),
                   c.items.as<CapItem>(), n_items, item_ticket, c.spans.as<int32_t>(), stride, tails ? d_line_off : nullptr,
                   tails ? c.recs.as<LineRec>() : nullptr, sep, tails ? c.tails.ext : nullptr, item_lines, interleave);
        tm.mark("k4b_bucket", 2);
        CapWalkParams W{};
        W.text = d_text;
        W.n_units = n_units;
        W.line_off = d_line_off;
        W.perm = c.perm.as<uint32_t>();
        W.items = c.items.as<CapItem>();
        W.n_items = n_items;
        W.item_ticket = item_ticket;
        W.img = c.capimg;
        W.cap = c.cap;
        W.span_stride = stride;
        W.smem_table_bytes = c.capimg.smem_table_bytes;
        if (const char* f = std::getenv("GORP_WALK_FLAGS")) W.flags = static_cast<uint32_t>(std::atoi(f));
        if (const char* f = std::getenv("GORP_CAP_FLAGS")) W.smem_table_bytes = (std::atoi(f) & 2) ? 0u : W.smem_table_bytes;
        W.ext_id = c.ext_id.as<int32_t>();
        W.spans = c.spans.as<int32_t>();
        W.hist = c.hist.as<unsigned long long>();
        if (tails) {
            TailWalkParams T{};
            T.text = d_text;
            T.n_units = n_units;
            T.line_off = d_line_off;
            T.perm = W.perm;
            T.items = W.items;
            T.n_items = n_items;
            T.item_ticket = tail_ticket;
            T.t = c.tails;
            T.n_ext = E;
            T.round_iters = c.tail_flush_every;
            T.lines_form = sep == 0 ? 1u : 0u;
            T.prefer_threads = interleave ? 512u : 0u;
            if (const char* f = std::getenv("GORP_TAIL_FLAGS")) T.flags = static_cast<uint32_t>(std::atoi(f));
            T.recs = c.recs.as<LineRec>();
            T.ext_id = W.ext_id;
            T.spans = W.spans;
            T.hist = W.hist;
            T.long_cap = static_cast<uint32_t>(n_units / kTailMaxLen + 2);
            c.long_lines.reserve(static_cast<size_t>(T.long_cap) * 4);
            T.long_lines = c.long_lines.as<uint32_t>();
            T.n_long = tail_ticket + 1;
            k4c_tailwalk(L, T);
            tm.mark("k4c_tailwalk", 2);
            W.skip_tails = c.tails.ext;
        }
        if (sep == 0) {  // List<String> form: the lines of extractions without a tail take the one-line-per-thread capture kernel
            if (c.tails.n_without > 0) {
                k4_tdfa_capture(L, c.cap, d_text, d_line_off, sep, n_lines, stride, c.ext_id.as<int32_t>(), c.spans.as<int32_t>(), c.tails.ext,
                                c.hist.as<unsigned long long>());
                tm.mark("k4_tdfa_capture", 1);
            }
        } else if (!tails || c.tails.n_without > 0) {
            k4b_capwalk(L, W);
            tm.mark("k4b_capwalk", 1);
        }
    } else if (!c.cap.match_only) {  // (also at stride 0: a definition without groups still has to fail the lines its regexes reject)
        if (sep == 1 && c.cap_fast.enabled && !c.force_general) {
            k4_tdfa_fast(L, c.cap_fast, c.cap, d_text, n_units, d_line_off, n_fast, stride, c.ext_id.as<int32_t>(), c.spans.as<int32_t>());
            if (n_fast < n_lines)
                k4_tdfa_capture(L, c.cap, d_text, d_line_off + n_fast, sep, 1, stride, c.ext_id.as<int32_t>() + n_fast,
                                c.spans.as<int32_t>() + static_cast<size_t>(n_fast) * stride);
            tm.mark("k4_tdfa_capture", n_fast < n_lines ? 2 : 1);
        } else {
            k4_tdfa_capture(L, c.cap, d_text, d_line_off, sep, n_lines, stride, c.ext_id.as<int32_t>(), c.spans.as<int32_t>());
            tm.mark("k4_tdfa_capture", 1);
        }
    } else {
        tm.mark("k4_tdfa_capture", 0);
    }
    if (!hist_done) {
        CK(cudaMemsetAsync(c.hist.p, 0, (c.n_ext + 2) * 8, stream));
        k3_histogram(L, c.ext_id.as<int32_t>(), n_lines, c.n_ext, c.hist.as<unsigned long long>());
        tm.mark("k3_histogram", 1);
    }
    CK(cudaGetLastError());
    if (out) {
        out->n_lines = n_lines;
        out->span_stride = static_cast<int32_t>(stride);
        out->d_ext_id = c.ext_id.as<int32_t>();
        out->d_line_off = d_line_off;
        out->d_spans = c.spans.as<int32_t>();
        out->d_histogram = c.hist.as<int64_t>();
        out->d_n_lines = d_n_lines;
    }
    return n_lines;
}

// ------------------------------------------------------------------ UTF-8 input: the steps around run_pipeline
// Shared by the host piece loop (run_pieces, on a staged piece) and the device-resident UTF-8 calls (on the caller's HBM).
// `bytes` is 16-byte aligned; the caller holds c.mu and has set the device.

// Text form, before the pipeline: UTF-16 units per tile + validation, scan, one host round trip ({decoded total, first
// malformed byte}, and the last byte when `last` is given), decode to `dst`. Returns the decoded total. `at` is the position
// of `bytes` in the caller's buffer (the error names a byte of the caller's buffer).
int64_t utf8_text_decode(DeviceCtx& c, const Launch& L, Timer& tm, const uint8_t* bytes, int64_t n, int64_t at, uint16_t* dst, uint8_t* last) {
    const int64_t tiles = utf8_tiles(n);
    c.tile_counts.reserve(static_cast<size_t>(tiles + 1) * 4);
    c.tile_base.reserve(static_cast<size_t>(tiles + 2) * 8);
    c.scan_scratch.reserve(static_cast<size_t>(tiles / 4096 + 8) * 8);
    c.scalars.reserve(128);
    unsigned long long* d_bad = reinterpret_cast<unsigned long long*>(c.scalars.as<int64_t>() + 6);
    unsigned long long bad = ~0ull;
    int64_t total = 0;
    CK(cudaMemsetAsync(d_bad, 0xFF, 8, L.stream));
    k_utf8_count(L, bytes, n, c.tile_counts.as<uint32_t>(), d_bad);
    scan_u32_to_i64(L, c.tile_counts.as<uint32_t>(), tiles, c.tile_base.as<int64_t>(), c.scan_scratch.as<int64_t>());
    tm.mark("utf8_count", 4);
    if (n > 0) CK(cudaMemcpyAsync(&total, c.tile_base.as<int64_t>() + tiles, 8, cudaMemcpyDeviceToHost, L.stream));
    CK(cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, L.stream));
    if (last && n > 0) CK(cudaMemcpyAsync(last, bytes + n - 1, 1, cudaMemcpyDeviceToHost, L.stream));
    CK(cudaStreamSynchronize(L.stream));
    if (bad != ~0ull)
        throw ArgError(strfmt("malformed UTF-8 at byte %lld (the input must be well-formed UTF-8)", static_cast<long long>(at + static_cast<int64_t>(bad))));
    k_utf8_write(L, bytes, n, c.tile_base.as<int64_t>(), dst);
    tm.mark("utf8_decode", 1);
    return total;
}

// Text form, after the pipeline: the byte '\n' index of `bytes` (built here because run_pipeline reuses tile_counts,
// tile_base, scan_scratch and nl_masks; line k of the bytes is line k of the decoded text: the same '\n' characters), then
// the rows `dr` moved from unit to byte offsets: out_off = byte line offsets + bias, out_spans = byte spans.
void utf8_text_rows(DeviceCtx& c, const Launch& L, Timer& tm, const uint8_t* bytes, int64_t n, bool ends_with_nl, const gorp_device_result& dr,
                    int64_t bias, uint32_t stride, int64_t* out_off, int32_t* out_spans) {
    const int64_t n_tiles = (n + kNlTile - 1) / kNlTile;
    c.tile_counts.reserve(static_cast<size_t>(n_tiles + 1) * 4);
    c.tile_base.reserve(static_cast<size_t>(n_tiles + 2) * 8);
    c.scan_scratch.reserve(static_cast<size_t>(n_tiles / 4096 + 8) * 8);
    c.nl_masks.reserve(static_cast<size_t>(n_tiles + 4) * 256 * 4);
    c.byte_off.reserve(static_cast<size_t>(dr.n_lines + 2) * 8);
    k_utf8_count_newlines_masks(L, bytes, n, c.tile_counts.as<uint32_t>(), c.nl_masks.as<uint32_t>());
    scan_u32_to_i64(L, c.tile_counts.as<uint32_t>(), n_tiles, c.tile_base.as<int64_t>(), c.scan_scratch.as<int64_t>());
    k1_scatter_masks(L, c.nl_masks.as<uint32_t>(), n, c.tile_base.as<int64_t>(), c.byte_off.as<int64_t>());
    tm.mark("utf8_nl_index", n > 0 ? 5 : 2);
    if (stride > 64) throw std::logic_error("result rows wider than 64 entries");  // (31 groups at most: 62)
    Utf8RowsParams P{};
    P.bytes = bytes;
    P.unit_off = dr.d_line_off;
    P.byte_off = c.byte_off.as<int64_t>();
    P.spans = dr.d_spans;
    P.n_lines = dr.n_lines;
    P.end_off = n + (ends_with_nl ? 0 : 1);
    P.bias = bias;
    P.stride = stride;
    P.out_off = out_off;
    P.out_spans = out_spans;
    k_utf8_rows(L, P);
    tm.mark("utf8_rows", 1);
}

// Lines form, before the pipeline: `bytes` holds bytes [at, at + n) of the caller's buffer, `d_off` the caller's n_lines + 1
// offsets (device memory). UTF-16 units per tile + slice prefixes + validation, scan, the strings' unit offsets (c.unit_off,
// relative to the piece) with the boundary check and, with `check_order`, the offset-order check; one host round trip;
// decode to `dst`. Returns the decoded total.
int64_t utf8_lines_decode(DeviceCtx& c, const Launch& L, Timer& tm, const uint8_t* bytes, int64_t n, int64_t at, const int64_t* d_off, int64_t n_lines,
                          uint16_t* dst, bool check_order) {
    const int64_t tiles = utf8_tiles(n);
    c.tile_counts.reserve(static_cast<size_t>(tiles + 1) * 4);
    c.tile_base.reserve(static_cast<size_t>(tiles + 2) * 8);
    c.scan_scratch.reserve(static_cast<size_t>(tiles / 4096 + 8) * 8);
    c.scalars.reserve(128);
    unsigned long long* d_bad = reinterpret_cast<unsigned long long*>(c.scalars.as<int64_t>() + 6);
    unsigned long long* d_order = check_order ? d_bad + 1 : nullptr;
    unsigned long long bad = ~0ull, order = ~0ull;
    int64_t total = 0;
    CK(cudaMemsetAsync(d_bad, 0xFF, check_order ? 16 : 8, L.stream));
    k_utf8_count(L, bytes, n, c.tile_counts.as<uint32_t>(), d_bad, c.slice_units.as<uint16_t>());
    scan_u32_to_i64(L, c.tile_counts.as<uint32_t>(), tiles, c.tile_base.as<int64_t>(), c.scan_scratch.as<int64_t>());
    tm.mark("utf8_count", 4);
    k_utf8_line_units(L, bytes, n, d_off, n_lines + 1, at, c.tile_base.as<int64_t>(), c.slice_units.as<uint16_t>(), c.unit_off.as<int64_t>(), d_bad,
                      d_order);
    tm.mark("utf8_line_units", 1);
    if (n > 0) CK(cudaMemcpyAsync(&total, c.tile_base.as<int64_t>() + tiles, 8, cudaMemcpyDeviceToHost, L.stream));
    CK(cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, L.stream));
    if (check_order) CK(cudaMemcpyAsync(&order, d_order, 8, cudaMemcpyDeviceToHost, L.stream));
    CK(cudaStreamSynchronize(L.stream));
    if (order != ~0ull) throw ArgError(strfmt("offsets must be non-decreasing (line %lld)", static_cast<long long>(order)));
    if (bad != ~0ull)
        throw ArgError(strfmt("malformed UTF-8 at byte %lld (every string must be well-formed UTF-8)", static_cast<long long>(at + static_cast<int64_t>(bad))));
    k_utf8_write(L, bytes, n, c.tile_base.as<int64_t>(), dst);
    tm.mark("utf8_decode", 1);
    return total;
}

// Lines form, after the pipeline: the rows `dr` moved back to the caller's byte offsets (out_off = a copy of d_off, or
// nullptr when the call returns d_off itself).
void utf8_lines_rows(const Launch& L, Timer& tm, const uint8_t* bytes, int64_t at, const int64_t* d_off, const gorp_device_result& dr, uint32_t stride,
                     int64_t* out_off, int32_t* out_spans) {
    if (stride > 64) throw std::logic_error("result rows wider than 64 entries");  // (31 groups at most: 62)
    Utf8RowsParams P{};
    P.bytes = bytes;
    P.unit_off = dr.d_line_off;
    P.byte_off = d_off;
    P.spans = dr.d_spans;
    P.n_lines = dr.n_lines;
    P.bias = at;
    P.stride = stride;
    P.out_off = out_off;
    P.out_spans = out_spans;
    k_utf8_rows(L, P, true);
    tm.mark("utf8_rows", 1);
}

// The UTF-8 device-resident calls write their rows in byte coordinates to acc_spans (and the text form its byte line
// offsets to acc_off): the accumulators of the host-buffer calls, idle outside those calls. utf8_rows_kernel reads the
// pipeline's unit rows while it writes, so it cannot write them in place.
void reserve_byte_rows(DeviceCtx& c, int64_t n_lines, uint32_t stride, bool offsets) {
    if (offsets) c.acc_off.reserve(static_cast<size_t>(n_lines + 2) * 8);
    c.acc_spans.reserve((static_cast<size_t>(n_lines) * stride + 4) * 4);
}

// ------------------------------------------------------------------ host-buffer calls: pieces, pipelining, devices
constexpr int64_t kPieceUnits = 32ll << 20;  // 64 MB of text per piece
constexpr int kTextPad = 32;                 // units in front of a staged piece (aligned chunk reads of the lines form)

struct Piece {
    int64_t u0, u1;  // units [u0, u1) of the caller's text
    int64_t l0, l1;  // lines [l0, l1) of the caller's offsets (lines form only)
};

// Cuts the batch into pieces of about kPieceUnits that end after a '\n' (text form) / at a string boundary (lines form).
template <class Unit>
std::vector<Piece> plan_pieces(const Unit* text, int64_t n_units, const int64_t* off, int64_t n_lines, int64_t piece_units) {
    std::vector<Piece> v;
    if (off) {
        int64_t l = 0;
        while (l < n_lines) {
            const int64_t* it = std::upper_bound(off + l + 1, off + n_lines + 1, off[l] + piece_units);
            int64_t l1 = (it - off) - 1;
            if (l1 <= l) l1 = l + 1;
            if (l1 > n_lines) l1 = n_lines;
            v.push_back({off[l], off[l1], l, l1});
            l = l1;
        }
        if (v.empty()) v.push_back({0, 0, 0, 0});
    } else {
        int64_t u = 0;
        while (u < n_units) {
            int64_t cut = std::min(u + piece_units, n_units);
            while (cut < n_units && text[cut - 1] != 0x0A) ++cut;
            v.push_back({u, cut, 0, 0});
            u = cut;
        }
        if (v.empty()) v.push_back({0, 0, 0, 0});
    }
    return v;
}

struct DeviceRun {  // what one device produced for its pieces
    int64_t n_rows = 0;
    int32_t stride = 0;
    std::string error;
    int status = GORP_OK;
};

// Processes pieces [p0, p1) on device context c. Rows accumulate in c.acc_*; when `hr` is given (single-device call) the
// rows of every finished piece are copied to the host arrays at once, overlapping the next pieces.
// `text8` (ISO-8859-1 bytes, text form only) replaces `text`: the bytes are staged and widened to UTF-16 on the device.
// `utf8`: the bytes are UTF-8, decoded on the device; offsets count UTF-16 units of the decoded text, or with `byte_coords`
// bytes of `text8` (then the pieces are independent, as for ISO-8859-1). `utf8` with `off` (always in byte coordinates): the
// caller's strings are bytes [off[i], off[i+1]) of `text8`; the piece is decoded at textbuf + kTextPad, its strings' unit
// offsets (relative to the piece) feed the lines form of the pipeline, and the rows go back to the caller's byte offsets.
// The caller holds c.mu (a multi-device call keeps every participating device locked until its rows are copied out).
// `keep_bytes` (UTF-8 in byte coordinates, for the value tables): the staged bytes of every piece are also copied to
// c.resident, which then holds bytes [pieces[p0].u0, pieces[p1 - 1].u1) of `text8`.
void run_pieces(gorp_engine* e, DeviceCtx& c, const uint16_t* text, const uint8_t* text8, bool utf8, bool byte_coords, const int64_t* off,
                const std::vector<Piece>& pieces, size_t p0, size_t p1, HostResult* hr, DeviceRun& run, bool keep_bytes = false) {
    CK(cudaSetDevice(c.device));
    // a device-resident call on another stream may still use the scratch: the kernels wait for it, and so do the staging
    // copies (the UTF-8 device calls decode into textbuf[0] and stage into bytebuf[0], which the first piece's copy overwrites)
    CK(cudaStreamWaitEvent(c.stream, c.ev_done, 0));
    CK(cudaStreamWaitEvent(c.s_in, c.ev_done, 0));
    Launch L{c.stream, c.sm_count};
    Timer tm(c, c.stream, false);  // (untimed: counts the launches)
    const size_t E2 = e->def.extractions.size() + 2;
    const uint32_t stride = e->match_only ? 0u : c.max_slots;
    int64_t units_total = 0, lines_total = 0;
    size_t max_units = 0, max_lines = 0;
    for (size_t k = p0; k < p1; ++k) {
        units_total += pieces[k].u1 - pieces[k].u0;
        lines_total += pieces[k].l1 - pieces[k].l0;
        max_units = std::max<size_t>(max_units, pieces[k].u1 - pieces[k].u0);
        max_lines = std::max<size_t>(max_lines, pieces[k].l1 - pieces[k].l0);
    }
    const int n_buf = p1 - p0 > 1 ? 2 : 1;
    for (int b = 0; b < n_buf; ++b) {
        c.textbuf[b].reserve((max_units + kTextPad + 64) * 2);
        if (text8) c.bytebuf[b].reserve(max_units + 64);
        if (off) c.offbuf[b].reserve((max_lines + 1) * 8);
    }
    if (keep_bytes) c.resident.reserve(static_cast<size_t>(units_total) + 64);
    if (off && utf8) {
        c.unit_off.reserve((max_lines + 1) * 8);
        c.slice_units.reserve((max_units / 16 + 1) * 2);
    }
    // row capacity: exact for the lines form; for the text form sized for the first piece from the running density
    // estimate, then (below) for the whole range from the density actually seen
    const int64_t units_first = pieces[p0].u1 - pieces[p0].u0;
    int64_t cap_rows = off ? lines_total : static_cast<int64_t>(static_cast<double>(units_first) * c.lines_per_unit * 1.25) + 4096;
    auto reserve_rows = [&](int64_t rows, int64_t keep) {
        c.acc_ext.grow_keep(static_cast<size_t>(rows + 1) * 4, static_cast<size_t>(keep) * 4, c.stream);
        c.acc_off.grow_keep(static_cast<size_t>(rows + 2) * 8, static_cast<size_t>(keep + 1) * 8, c.stream);
        c.acc_spans.grow_keep((static_cast<size_t>(rows) * stride + 4) * 4, static_cast<size_t>(keep) * stride * 4, c.stream);
        if (hr) {
            hr->reserve(0, static_cast<size_t>(rows + 1) * 4, static_cast<size_t>(keep) * 4);
            hr->reserve(1, static_cast<size_t>(rows + 2) * 8, static_cast<size_t>(keep + 1) * 8);
            hr->reserve(2, (static_cast<size_t>(rows) * stride + 4) * 4, static_cast<size_t>(keep) * stride * 4);
        }
    };
    reserve_rows(cap_rows, 0);
    c.acc_hist.reserve(E2 * 8);
    CK(cudaMemsetAsync(c.acc_hist.p, 0, E2 * 8, c.stream));

    auto stage = [&](size_t k) {  // H2D of piece k on s_in
        const Piece& pc = pieces[k];
        const int b = static_cast<int>((k - p0) & 1);
        const int64_t units = pc.u1 - pc.u0;
        const int64_t lead = off ? kTextPad + (pc.u0 & 15) : 0;  // keeps (device address - unit index) a multiple of 32 bytes
        if (k >= p0 + 2) CK(cudaStreamWaitEvent(c.s_in, c.ev_free[b], 0));  // the gather of piece k-2 still reads this buffer's offsets
        if (units && text8)
            CK(cudaMemcpyAsync(c.bytebuf[b].p, text8 + pc.u0, static_cast<size_t>(units), cudaMemcpyHostToDevice, c.s_in));
        else if (units)
            CK(cudaMemcpyAsync(c.textbuf[b].as<uint16_t>() + lead, text + pc.u0, static_cast<size_t>(units) * 2, cudaMemcpyHostToDevice, c.s_in));
        if (off)
            CK(cudaMemcpyAsync(c.offbuf[b].p, off + pc.l0, static_cast<size_t>(pc.l1 - pc.l0 + 1) * 8, cudaMemcpyHostToDevice, c.s_in));
        CK(cudaEventRecord(c.ev_in[b], c.s_in));
    };

    int64_t rows = 0;
    int64_t utf8_base = 0;  // UTF-16 units decoded from the pieces before this one (UTF-8 input: offsets are in decoded units)
    stage(p0);
    for (size_t k = p0; k < p1; ++k) {
        const Piece& pc = pieces[k];
        const int b = static_cast<int>((k - p0) & 1);
        if (k + 1 < p1) stage(k + 1);  // the other buffer: its previous piece was computed (this thread waited for it)
        CK(cudaStreamWaitEvent(c.stream, c.ev_in[b], 0));
        const int64_t units = pc.u1 - pc.u0;
        if (keep_bytes && units)
            CK(cudaMemcpyAsync(c.resident.as<uint8_t>() + (pc.u0 - pieces[p0].u0), c.bytebuf[b].p, static_cast<size_t>(units), cudaMemcpyDeviceToDevice,
                               c.stream));
        int64_t piece_bias = pc.u0;  // what turns the piece's line offsets into offsets of the whole batch
        gorp_device_result dr{};
        int64_t nl;
        if (off && utf8) {
            // UTF-8 strings (the host checked the offsets): decoded behind the lines-form padding, then the lines form over
            // the decoded piece
            const int64_t n_lines_piece = pc.l1 - pc.l0;
            uint16_t* piece_text = c.textbuf[b].as<uint16_t>() + kTextPad;  // (device address - unit index) a multiple of 32 bytes
            const int64_t total = utf8_lines_decode(c, L, tm, c.bytebuf[b].as<uint8_t>(), units, pc.u0, c.offbuf[b].as<int64_t>(), n_lines_piece,
                                                    piece_text, false);
            nl = run_pipeline(c, piece_text, total, c.unit_off.as<int64_t>(), n_lines_piece, c.stream, tm, &dr);
        } else if (off) {
            const uint16_t* vbase = c.textbuf[b].as<uint16_t>() + kTextPad + (pc.u0 & 15) - pc.u0;  // text[i] lives at vbase + i
            nl = run_pipeline(c, vbase, pc.u1, c.offbuf[b].as<int64_t>(), pc.l1 - pc.l0, c.stream, tm, &dr);  // text[i] valid for i < u1
        } else {
            int64_t n_units_piece = units;
            if (text8 && utf8) {
                n_units_piece = utf8_text_decode(c, L, tm, c.bytebuf[b].as<uint8_t>(), units, pc.u0, c.textbuf[b].as<uint16_t>(), nullptr);
            } else if (text8) {
                k_widen_latin1(L, c.bytebuf[b].as<uint8_t>(), c.textbuf[b].as<uint16_t>(), units);
                c.launches += 1;
            }
            nl = run_pipeline(c, c.textbuf[b].as<uint16_t>(), n_units_piece, nullptr, 0, c.stream, tm, &dr);
            if (utf8 && !byte_coords) {
                piece_bias = utf8_base;
                utf8_base += n_units_piece;
            }
        }
        if (rows + nl > cap_rows) {  // the density estimate was too low: grow, keeping the rows gathered so far
            if (hr) CK(cudaStreamSynchronize(c.s_out));
            cap_rows = std::max<int64_t>(rows + nl, static_cast<int64_t>(static_cast<double>(rows + nl) / std::max<int64_t>(pc.u1 - pieces[p0].u0, 1) *
                                                                         static_cast<double>(units_total) * 1.1) + 4096);
            reserve_rows(cap_rows, rows);
        }
        // gather: rows [rows, rows + nl) of the batch
        if (nl) CK(cudaMemcpyAsync(c.acc_ext.as<int32_t>() + rows, dr.d_ext_id, static_cast<size_t>(nl) * 4, cudaMemcpyDeviceToDevice, c.stream));
        if (off && utf8) {
            // rows back to the caller's byte offsets (line_off is a copy of the caller's offsets)
            utf8_lines_rows(L, tm, c.bytebuf[b].as<uint8_t>(), pc.u0, c.offbuf[b].as<int64_t>(), dr, stride, c.acc_off.as<int64_t>() + rows,
                            c.acc_spans.as<int32_t>() + static_cast<size_t>(rows) * stride);
        } else if (utf8 && byte_coords) {
            utf8_text_rows(c, L, tm, c.bytebuf[b].as<uint8_t>(), units, units == 0 || text8[pc.u1 - 1] == 0x0A, dr, piece_bias, stride,
                           c.acc_off.as<int64_t>() + rows, c.acc_spans.as<int32_t>() + static_cast<size_t>(rows) * stride);
        } else {
            k_bias_copy(L, c.acc_off.as<int64_t>() + rows, dr.d_line_off, nl + 1, off ? 0 : piece_bias);
            if (nl && stride)
                CK(cudaMemcpyAsync(c.acc_spans.as<int32_t>() + static_cast<size_t>(rows) * stride, dr.d_spans, static_cast<size_t>(nl) * stride * 4,
                                   cudaMemcpyDeviceToDevice, c.stream));
            c.launches += 1;
        }
        k_accumulate(L, c.acc_hist.as<int64_t>(), dr.d_histogram, static_cast<int>(E2));
        c.launches += 1;
        CK(cudaEventRecord(c.ev_free[b], c.stream));
        if (hr) {
            CK(cudaEventRecord(c.ev_rows, c.stream));
            CK(cudaStreamWaitEvent(c.s_out, c.ev_rows, 0));
            if (nl) CK(cudaMemcpyAsync(static_cast<int32_t*>(hr->p[0]) + rows, c.acc_ext.as<int32_t>() + rows, static_cast<size_t>(nl) * 4, cudaMemcpyDeviceToHost, c.s_out));
            CK(cudaMemcpyAsync(static_cast<int64_t*>(hr->p[1]) + rows, c.acc_off.as<int64_t>() + rows, static_cast<size_t>(nl + 1) * 8, cudaMemcpyDeviceToHost, c.s_out));
            if (nl && stride)
                CK(cudaMemcpyAsync(static_cast<int32_t*>(hr->p[2]) + static_cast<size_t>(rows) * stride, c.acc_spans.as<int32_t>() + static_cast<size_t>(rows) * stride,
                                   static_cast<size_t>(nl) * stride * 4, cudaMemcpyDeviceToHost, c.s_out));
        }
        rows += nl;
    }
    if (hr) {
        hr->reserve(3, E2 * 8);
        CK(cudaStreamWaitEvent(c.s_out, c.ev_rows, 0));
        CK(cudaMemcpyAsync(hr->p[3], c.acc_hist.p, E2 * 8, cudaMemcpyDeviceToHost, c.stream));
        CK(cudaStreamSynchronize(c.stream));
        CK(cudaStreamSynchronize(c.s_out));
    } else {
        CK(cudaStreamSynchronize(c.stream));
    }
    CK(cudaEventRecord(c.ev_done, c.stream));
    run.n_rows = rows;
    run.stride = static_cast<int32_t>(stride);
}

// Host copy of the layout that build_tables leaves in c.tb_*.
struct TablesBuilt {
    std::vector<TableLayout> lay;   // [E + 1]; entry E holds the totals
    std::vector<int64_t> stats;     // [2 * columns]: value units, nulls
    std::vector<int64_t> col_info;  // [2 * columns + 2]: first entry of the column in the offset scan, byte offset of its data
    int64_t n_cols = 0;
};

// The value tables (kernels/tables.cu, DESIGN.md §5.5) of rows `r` of context c, values read from `text` (unit_bytes per
// unit) at line_off + span: row indexes in c.tb_rows, offsets in c.tb_offs (from 0 in every column), values in c.tb_data,
// bitmaps in c.tb_valid, positions in `b`. Four stages on `st`, one host round trip (the per-column totals size the values).
void build_tables(gorp_engine* e, DeviceCtx& c, cudaStream_t st, Timer& tm, const gorp_device_result& r, const void* text, int ub,
                  TablesBuilt& b) {
    Launch L{st, c.sm_count};
    const uint32_t E = c.n_ext;
    const int64_t n = r.n_lines;
    const uint32_t stride = static_cast<uint32_t>(r.span_stride);
    int64_t n_cols = 0;  // columns of all tables
    for (const auto& x : e->def.extractions) n_cols += stride ? x.n_groups : 0;
    // 1. rank: stable partition of the matched lines by extraction
    const int64_t tile = tables_tile_lines(E), n_tiles = std::max<int64_t>(1, (n + tile - 1) / tile), cells = n_tiles * E;
    c.tb_counts.reserve(static_cast<size_t>(cells) * 4 + 64);
    c.tb_starts.reserve(static_cast<size_t>(cells + 1) * 8 + 64);
    c.tb_layout.reserve((E + 1) * sizeof(TableLayout));
    c.tb_rows.reserve(static_cast<size_t>(n + 8 * E + 8) * 8);
    c.tb_stats.reserve(static_cast<size_t>(n_cols) * 16 + 64);
    TableLayout* lay = c.tb_layout.as<TableLayout>();
    k_tables_count(L, r.d_ext_id, n, E, tile, n_tiles, c.tb_counts.as<uint32_t>());
    c.tb_scan.reserve(static_cast<size_t>(cells / 4096 + 8) * 8);
    scan_u32_to_i64(L, c.tb_counts.as<uint32_t>(), cells, c.tb_starts.as<int64_t>(), c.tb_scan.as<int64_t>());
    k_tables_layout(L, c.tb_starts.as<int64_t>(), n_tiles, E, c.d_slots, stride != 0, lay);
    k_tables_scatter(L, r.d_ext_id, n, E, tile, n_tiles, c.tb_starts.as<int64_t>(), lay, c.tb_rows.as<int64_t>());
    CK(cudaGetLastError());
    tm.mark("tables_rank", 6);
    // 2. lengths, validity, per-column totals and null counts (sized for every line in the widest extraction)
    const int64_t slots_ub = n * (stride / 2) + 8 * n_cols + 8, words_ub = n * (stride / 2) / 32 + 17 * n_cols + 16;
    c.tb_lens.reserve(static_cast<size_t>(slots_ub) * 4);
    c.tb_valid.reserve(static_cast<size_t>(words_ub) * 4);
    CK(cudaMemsetAsync(c.tb_valid.p, 0, static_cast<size_t>(words_ub) * 4, st));
    if (n_cols) CK(cudaMemsetAsync(c.tb_stats.p, 0, static_cast<size_t>(n_cols) * 16, st));
    k_tables_len(L, lay, E, c.tb_rows.as<int64_t>(), r.d_spans, stride, c.tb_lens.as<uint32_t>(), c.tb_valid.as<uint32_t>(),
                 c.tb_stats.as<unsigned long long>());
    CK(cudaGetLastError());
    tm.mark("tables_len", 1);
    // the one round trip: the layout and the column totals
    b.lay.assign(E + 1, TableLayout{});
    b.stats.assign(static_cast<size_t>(n_cols) * 2, 0);
    CK(cudaMemcpyAsync(b.lay.data(), lay, (E + 1) * sizeof(TableLayout), cudaMemcpyDeviceToHost, st));
    if (n_cols) CK(cudaMemcpyAsync(b.stats.data(), c.tb_stats.p, b.stats.size() * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (b.lay[E].col_base != n_cols) throw std::runtime_error("value tables: column count mismatch");
    // 3. offsets: one scan over the lengths of every column; 4. gather into 64-byte aligned columns
    const int64_t n_off = b.lay[E].off_base;
    b.n_cols = n_cols;
    b.col_info.assign(static_cast<size_t>(n_cols) * 2 + 2, 0);
    int64_t flat = 0, data_bytes = 0;
    for (int64_t k = 0; k < n_cols; ++k) {
        b.col_info[2 * k] = flat;
        b.col_info[2 * k + 1] = data_bytes;
        flat += b.stats[2 * k];
        data_bytes += (b.stats[2 * k] * ub + 63) / 64 * 64;
    }
    c.tb_offs.reserve(static_cast<size_t>(n_off + 1) * 8 + 64);
    c.tb_scan.reserve(static_cast<size_t>(n_off / 4096 + 8) * 8);
    scan_u32_to_i64(L, c.tb_lens.as<uint32_t>(), n_off, c.tb_offs.as<int64_t>(), c.tb_scan.as<int64_t>());
    CK(cudaGetLastError());
    tm.mark("tables_scan", 3);
    c.tb_colinfo.reserve(b.col_info.size() * 8);
    // (pageable: the copy has been staged by the time cudaMemcpyAsync returns)
    CK(cudaMemcpyAsync(c.tb_colinfo.p, b.col_info.data(), b.col_info.size() * 8, cudaMemcpyHostToDevice, st));
    c.tb_data.reserve(static_cast<size_t>(data_bytes) + 64);
    k_tables_gather(L, lay, E, c.tb_rows.as<int64_t>(), r.d_line_off, r.d_spans, stride, text, ub, c.tb_lens.as<uint32_t>(),
                    c.tb_offs.as<int64_t>(), c.tb_colinfo.as<int64_t>(), c.tb_data.as<uint8_t>());
    CK(cudaGetLastError());
    tm.mark("tables_gather", 1);
}

// The tables of a UTF-8 host call in pinned memory of hr: device d < G built the tables of its rows (bt[d], lines
// [base[d], base[d + 1]) of the result); table e takes device d's rows after those of the devices before it. On one device
// the buffers are copied as they are. On several, device d first adds its line base to its row indexes and the column's
// value base to its offsets, and moves its bitmaps to the bit position of its first row (k_tables_rebase); where that
// position is not a multiple of 8, the first byte is ORed into the byte the previous device wrote, here on the host. The
// copies of all devices run at once; returns when they are done.
void merge_tables(gorp_engine* e, size_t G, const std::vector<TablesBuilt>& bt, const std::vector<int64_t>& base, HostResult& hr) {
    const size_t E = e->def.extractions.size();
    const int64_t n_cols = bt[0].n_cols;
    auto up64 = [](int64_t x) { return (x + 63) / 64 * 64; };
    // positions in the host buffers (bytes) and every device's row and value bases
    std::vector<int64_t> n_rows(E, 0), row_at(E), col_rows(static_cast<size_t>(n_cols)), off_at(static_cast<size_t>(n_cols)),
        data_at(static_cast<size_t>(n_cols)), valid_at(static_cast<size_t>(n_cols)), values(static_cast<size_t>(n_cols), 0),
        nulls(static_cast<size_t>(n_cols), 0);
    std::vector<int64_t> row_base(G * E), value_base(G * static_cast<size_t>(n_cols));
    for (size_t d = 0; d < G; ++d)
        for (size_t t = 0; t < E; ++t) {
            row_base[d * E + t] = n_rows[t];
            n_rows[t] += bt[d].lay[t].n_rows;
        }
    for (size_t d = 0; d < G; ++d)
        for (int64_t k = 0; k < n_cols; ++k) {
            value_base[d * n_cols + k] = values[k];
            values[k] += bt[d].stats[2 * k];
            nulls[k] += bt[d].stats[2 * k + 1];
        }
    int64_t rows_bytes = 0, off_bytes = 0, data_bytes = 0, valid_bytes = 0;
    for (size_t t = 0; t < E; ++t) {
        row_at[t] = rows_bytes;
        rows_bytes += up64(n_rows[t] * 8);
        const TableLayout& x = bt[0].lay[t];
        for (int64_t k = x.col_base; k < x.col_base + x.n_cols; ++k) {
            col_rows[k] = n_rows[t];
            off_at[k] = off_bytes;
            off_bytes += up64((n_rows[t] + 1) * 8);
            data_at[k] = data_bytes;
            data_bytes += up64(values[k]);
            valid_at[k] = valid_bytes;
            valid_bytes += up64((n_rows[t] + 7) / 8);
        }
    }
    // (behind the bitmaps: the first byte of every device's shifted bitmaps, ORed in below)
    const int64_t side_at = valid_bytes;
    hr.reserve(4, static_cast<size_t>(rows_bytes) + 64);
    hr.reserve(5, static_cast<size_t>(off_bytes) + 64);
    hr.reserve(6, static_cast<size_t>(data_bytes) + 64);
    hr.reserve(7, static_cast<size_t>(valid_bytes + static_cast<int64_t>(G) * n_cols) + 64);
    uint8_t* h_rows = static_cast<uint8_t*>(hr.p[4]);
    uint8_t* h_off = static_cast<uint8_t*>(hr.p[5]);
    uint8_t* h_data = static_cast<uint8_t*>(hr.p[6]);
    uint8_t* h_valid = static_cast<uint8_t*>(hr.p[7]);
    for (size_t d = 0; d < G; ++d) {
        DeviceCtx& c = *e->devs[d];
        CK(cudaSetDevice(c.device));
        const TablesBuilt& b = bt[d];
        auto dev_rows = [&](size_t t) { return c.tb_rows.as<int64_t>() + b.lay[t].row_base; };
        auto dev_off = [&](size_t t, int64_t k) { return c.tb_offs.as<int64_t>() + b.lay[t].off_base + (k - b.lay[t].col_base) * b.lay[t].seg; };
        auto dev_valid = [&](size_t t, int64_t k) {
            return reinterpret_cast<uint8_t*>(c.tb_valid.as<uint32_t>() + b.lay[t].valid_base + (k - b.lay[t].col_base) * b.lay[t].vwords);
        };
        // the rebase: row indexes and offsets in place, bitmaps into tb_stage
        std::vector<RebaseJob> jobs;
        std::vector<int64_t> stage_at(static_cast<size_t>(n_cols), -1);
        int64_t blocks = 0, stage_bytes = 0;
        auto add_job = [&](RebaseJob j) {
            j.first_block = blocks;
            blocks += tables_rebase_blocks(j);
            jobs.push_back(j);
        };
        for (size_t t = 0; t < E; ++t) {
            const TableLayout& x = b.lay[t];
            const int64_t rb = row_base[d * E + t];
            if (x.n_rows && base[d]) add_job({dev_rows(t), dev_rows(t), x.n_rows, base[d], 0, 0});
            for (int64_t k = x.col_base; k < x.col_base + x.n_cols; ++k) {
                if (value_base[d * n_cols + k]) add_job({dev_off(t, k), dev_off(t, k), x.n_rows + 1, value_base[d * n_cols + k], 0, 0});
                if (x.n_rows && rb % 8) {
                    stage_at[k] = stage_bytes;
                    stage_bytes += up64((x.n_rows + rb % 8 + 7) / 8);
                }
            }
        }
        c.tb_stage.reserve(static_cast<size_t>(stage_bytes) + 64);
        for (size_t t = 0; t < E; ++t)
            for (int64_t k = b.lay[t].col_base; k < b.lay[t].col_base + b.lay[t].n_cols; ++k)
                if (stage_at[k] >= 0)
                    add_job({dev_valid(t, k), c.tb_stage.as<uint8_t>() + stage_at[k], b.lay[t].n_rows, 0, row_base[d * E + t] % 8, 0});
        if (!jobs.empty()) {
            c.tb_jobs.reserve(jobs.size() * sizeof(RebaseJob));
            CK(cudaMemcpyAsync(c.tb_jobs.p, jobs.data(), jobs.size() * sizeof(RebaseJob), cudaMemcpyHostToDevice, c.stream));  // (pageable)
            k_tables_rebase(Launch{c.stream, c.sm_count}, c.tb_jobs.as<RebaseJob>(), static_cast<uint32_t>(jobs.size()), blocks);
            CK(cudaGetLastError());
            c.launches += 1;
        }
        // the copies to the host buffers
        auto d2h = [&](void* dst, const void* src, int64_t bytes) {
            if (bytes > 0) CK(cudaMemcpyAsync(dst, src, static_cast<size_t>(bytes), cudaMemcpyDeviceToHost, c.stream));
        };
        for (size_t t = 0; t < E; ++t) {
            const TableLayout& x = b.lay[t];
            const int64_t rb = row_base[d * E + t];
            d2h(h_rows + row_at[t] + rb * 8, dev_rows(t), x.n_rows * 8);
            for (int64_t k = x.col_base; k < x.col_base + x.n_cols; ++k) {
                // offsets: entries [rb, rb + n) (the last device also the closing entry); values; bitmaps
                d2h(h_off + off_at[k] + rb * 8, dev_off(t, k), (x.n_rows + (d + 1 == G ? 1 : 0)) * 8);
                d2h(h_data + data_at[k] + value_base[d * n_cols + k], c.tb_data.as<uint8_t>() + b.col_info[2 * k + 1], b.stats[2 * k]);
                if (stage_at[k] < 0) {
                    d2h(h_valid + valid_at[k] + rb / 8, dev_valid(t, k), (x.n_rows + 7) / 8);
                } else {
                    const uint8_t* s = c.tb_stage.as<uint8_t>() + stage_at[k];
                    d2h(h_valid + side_at + d * n_cols + k, s, 1);
                    d2h(h_valid + valid_at[k] + rb / 8 + 1, s + 1, (x.n_rows + rb % 8 + 7) / 8 - 1);
                }
            }
        }
    }
    for (size_t d = 0; d < G; ++d) {
        CK(cudaSetDevice(e->devs[d]->device));
        CK(cudaStreamSynchronize(e->devs[d]->stream));
        CK(cudaEventRecord(e->devs[d]->ev_done, e->devs[d]->stream));
    }
    hr.tables.reset(E, n_cols);
    for (size_t t = 0; t < E; ++t) {
        const TableLayout& x = bt[0].lay[t];
        for (int64_t k = x.col_base; k < x.col_base + x.n_cols; ++k) {
            uint8_t* v = h_valid + valid_at[k];
            for (size_t d = 1; d < G; ++d)
                if (bt[d].lay[t].n_rows && row_base[d * E + t] % 8) v[row_base[d * E + t] / 8] |= h_valid[side_at + d * n_cols + k];
            const int64_t used = (n_rows[t] + 7) / 8;
            std::memset(v + used, 0, static_cast<size_t>(up64(used) - used));
            hr.tables.offsets[k] = reinterpret_cast<const int64_t*>(h_off + off_at[k]);
            hr.tables.data[k] = h_data + data_at[k];
            hr.tables.valid[k] = v;
            hr.tables.nulls[k] = nulls[k];
        }
        hr.tables.set_table(t, n_rows[t], reinterpret_cast<const int64_t*>(h_rows + row_at[t]), x.col_base, x.n_cols);
    }
}

int extract_host(gorp_engine* e, const uint16_t* text, const uint8_t* text8, int64_t n_units, const int64_t* off, int64_t n_lines,
                 gorp_result* out, bool utf8 = false, bool byte_coords = false, gorp_device_tables* tables = nullptr) {
    if (!e || !out || (!text && !text8 && n_units > 0) || n_units < 0 || n_lines < 0) return fail(GORP_E_ARG, "bad argument");
    if (e->devs.empty()) return fail(GORP_E_CUDA, "engine has no CUDA device");
    return guarded([&]() -> int {
        // byte inputs (ISO-8859-1 / UTF-8) move half the bytes per unit: 4x the units per piece keeps the per-piece overhead
        // (a dozen small launches and one host round trip) below the copy time — measured on config #2 (profiles/README.md
        // round 2): 149 -> 132 ms per 100 M lines of Latin-1 input
        int64_t piece_units = text8 ? 4 * kPieceUnits : kPieceUnits;
        // (the lines form pays two copies and a longer kernel chain per piece: larger pieces once the batch has 16 of them)
        if (off && n_lines > 0 && !text8) piece_units = std::min<int64_t>(4 * kPieceUnits, std::max<int64_t>(kPieceUnits, n_units / 16));
        if (const char* f = std::getenv("GORP_PIECE_UNITS")) piece_units = std::max<int64_t>(std::atoll(f), 1024);
        const std::vector<Piece> pieces = text8 ? plan_pieces(text8, n_units, off, n_lines, piece_units) : plan_pieces(text, n_units, off, n_lines, piece_units);
        std::unique_ptr<HostResult> hr;
        {
            std::lock_guard<std::mutex> pl(e->pool_mu);
            if (!e->pool.empty()) {
                hr = std::move(e->pool.back());
                e->pool.pop_back();
            }
        }
        if (!hr) {
            hr = std::make_unique<HostResult>();
            hr->numa_node = e->devs[0]->numa_node;
        }
        const size_t E2 = e->def.extractions.size() + 2;
        // UTF-8 input with offsets in decoded units: those are known only piece after piece — one device per call
        // (in byte coordinates the host knows every piece's position, as for ISO-8859-1)
        const size_t G = utf8 && !byte_coords ? 1 : std::min(e->devs.size(), pieces.size());
        int64_t nl = 0;
        int32_t stride = 0;
        DeviceGuard restore_device;
        // value tables (UTF-8 in byte coordinates): every device builds the tables of its rows over its resident bytes
        auto device_tables = [&](DeviceCtx& c, const DeviceRun& run, size_t p0, TablesBuilt& b) {
            gorp_device_result r{};
            r.n_lines = run.n_rows;
            r.span_stride = run.stride;
            r.d_ext_id = c.acc_ext.as<int32_t>();
            r.d_line_off = c.acc_off.as<int64_t>();
            r.d_spans = c.acc_spans.as<int32_t>();
            Timer tm(c, c.stream, false);  // (untimed: counts the launches)
            build_tables(e, c, c.stream, tm, r, c.resident.as<uint8_t>() - pieces[p0].u0, 1, b);
        };
        if (G <= 1) {
            DeviceRun run;
            CtxLock lock(*e->devs[0]);
            run_pieces(e, *e->devs[0], text, text8, utf8, byte_coords, off, pieces, 0, pieces.size(), hr.get(), run, tables != nullptr);
            nl = run.n_rows;
            stride = run.stride;
            if (tables) {
                std::vector<TablesBuilt> bt(1);
                device_tables(*e->devs[0], run, 0, bt[0]);
                merge_tables(e, 1, bt, {0}, *hr);
            }
        } else {
            // contiguous ranges of pieces per device (lines shard as contiguous ranges: no data crosses devices); one
            // host thread per device; the rows are copied out once every device's row base is known
            // every participating device stays locked (in device order) from the first kernel to the last row copied out:
            // a concurrent call on the same engine can neither overwrite the accumulators nor free them in between
            std::vector<CtxLock> locks;
            for (size_t d = 0; d < G; ++d) locks.emplace_back(*e->devs[d]);
            std::vector<DeviceRun> runs(G);
            std::vector<TablesBuilt> bt(tables ? G : 0);
            std::vector<size_t> first(G + 1);
            for (size_t d = 0; d <= G; ++d) first[d] = pieces.size() * d / G;
            std::vector<std::thread> th;
            for (size_t d = 0; d < G; ++d)
                th.emplace_back([&, d]() {
                    runs[d].status = guarded([&]() -> int {
                        run_pieces(e, *e->devs[d], text, text8, utf8, byte_coords, off, pieces, first[d], first[d + 1], nullptr, runs[d],
                                   tables != nullptr);
                        if (tables) device_tables(*e->devs[d], runs[d], first[d], bt[d]);
                        return GORP_OK;
                    });
                    if (runs[d].status != GORP_OK) runs[d].error = g_error;
                });
            for (auto& t : th) t.join();
            // (the first device that failed: for malformed UTF-8 that is the lowest offending byte, the ranges being in byte order)
            for (size_t d = 0; d < G; ++d)
                if (runs[d].status != GORP_OK) return fail(runs[d].status, runs[d].error);
            std::vector<int64_t> base(G + 1, 0);
            for (size_t d = 0; d < G; ++d) base[d + 1] = base[d] + runs[d].n_rows;
            nl = base[G];
            stride = runs[0].stride;
            hr->reserve(0, static_cast<size_t>(nl + 1) * 4);
            hr->reserve(1, static_cast<size_t>(nl + 2) * 8);
            hr->reserve(2, (static_cast<size_t>(nl) * stride + 4) * 4);
            hr->reserve(3, E2 * 8);
            std::vector<int64_t> hist(G * E2);
            for (size_t d = 0; d < G; ++d) {
                DeviceCtx& c = *e->devs[d];
                CK(cudaSetDevice(c.device));
                const int64_t n = runs[d].n_rows;
                if (n) CK(cudaMemcpyAsync(static_cast<int32_t*>(hr->p[0]) + base[d], c.acc_ext.p, static_cast<size_t>(n) * 4, cudaMemcpyDeviceToHost, c.stream));
                CK(cudaMemcpyAsync(static_cast<int64_t*>(hr->p[1]) + base[d], c.acc_off.p, static_cast<size_t>(n + (d + 1 == G ? 1 : 0)) * 8, cudaMemcpyDeviceToHost, c.stream));
                if (n && stride)
                    CK(cudaMemcpyAsync(static_cast<int32_t*>(hr->p[2]) + static_cast<size_t>(base[d]) * stride, c.acc_spans.p, static_cast<size_t>(n) * stride * 4,
                                       cudaMemcpyDeviceToHost, c.stream));
                CK(cudaMemcpyAsync(hist.data() + d * E2, c.acc_hist.p, E2 * 8, cudaMemcpyDeviceToHost, c.stream));
            }
            if (tables) merge_tables(e, G, bt, base, *hr);  // (its copies run alongside those of the rows)
            for (size_t d = 0; d < G; ++d) {
                CK(cudaSetDevice(e->devs[d]->device));
                CK(cudaStreamSynchronize(e->devs[d]->stream));
            }
            int64_t* h = static_cast<int64_t*>(hr->p[3]);
            for (size_t i = 0; i < E2; ++i) {
                h[i] = 0;
                for (size_t d = 0; d < G; ++d) h[i] += hist[d * E2 + i];
            }
        }
        out->n_lines = nl;
        out->n_extractions = static_cast<int32_t>(e->def.extractions.size());
        out->span_stride = stride;
        out->ext_id = static_cast<const int32_t*>(hr->p[0]);
        out->line_off = static_cast<const int64_t*>(hr->p[1]);
        out->spans = static_cast<const int32_t*>(hr->p[2]);
        out->histogram = static_cast<const int64_t*>(hr->p[3]);
        if (tables) hr->tables.describe(tables, 1);
        out->owner = hr.release();
        return GORP_OK;
    });
}

// ---- blob walking without copies (for the introspection entry points)
struct BlobView {
    const uint8_t* base;
    size_t len;
    uint32_t S, C, E;
    size_t classmap, trans, acc_first, acc_off, acc_list, ext0;
};

bool view_blob(const void* blob, size_t len, BlobView& v) {
    // parse_blob validates everything (magic, checksum, ranges); the view only records offsets
    CompiledDefinition d = parse_blob(blob, len);
    v.base = static_cast<const uint8_t*>(blob);
    v.len = len;
    v.S = d.dfa.n_states;
    v.C = d.dfa.n_classes;
    v.E = static_cast<uint32_t>(d.extractions.size());
    v.classmap = 40;
    v.trans = v.classmap + 65536 * 2;
    v.acc_first = v.trans + static_cast<size_t>(v.S) * v.C * 4;
    v.acc_off = v.acc_first + static_cast<size_t>(v.S) * 4;
    v.acc_list = v.acc_off + static_cast<size_t>(v.S + 1) * 4;
    v.ext0 = v.acc_list + d.dfa.accept_list.size() * 4;
    return true;
}

struct StrRef {
    const uint16_t* p;
    uint32_t n;
};

size_t read_str(const BlobView& v, size_t at, StrRef& s) {
    uint32_t n;
    std::memcpy(&n, v.base + at, 4);
    s.p = reinterpret_cast<const uint16_t*>(v.base + at + 4);
    s.n = n;
    size_t next = at + 4 + static_cast<size_t>(n) * 2;
    return (next + 3) & ~size_t(3);
}

// walks to extraction `index`; fills info and (optionally) the k-th extractor name
void locate_extraction(const BlobView& v, uint32_t index, gorp_extraction_info* info, uint32_t k, StrRef* name_k) {
    size_t at = v.ext0;
    for (uint32_t e = 0;; ++e) {
        uint32_t groups;
        std::memcpy(&groups, v.base + at, 4);
        at += 4;
        StrRef name, autom, jdk;
        at = read_str(v, at, name);
        at = read_str(v, at, autom);
        at = read_str(v, at, jdk);
        uint32_t nn;
        std::memcpy(&nn, v.base + at, 4);
        at += 4;
        for (uint32_t j = 0; j < nn; ++j) {
            StrRef s;
            at = read_str(v, at, s);
            if (e == index && name_k && j == k) *name_k = s;
        }
        uint32_t jl;
        std::memcpy(&jl, v.base + at, 4);
        at += 4;
        const char* json = reinterpret_cast<const char*>(v.base + at);
        at = (at + jl + 3) & ~size_t(3);
        if (e == index) {
            if (info) {
                info->n_groups = groups;
                info->n_extractor_names = nn;
                info->name = name.p;
                info->name_len = name.n;
                info->automaton_regex = autom.p;
                info->automaton_regex_len = autom.n;
                info->jdk_regex = jdk.p;
                info->jdk_regex_len = jdk.n;
                info->append_json = json;
                info->append_json_len = jl;
            }
            return;
        }
    }
}

int export_blob(const CompiledDefinition& d, bool match_only, void** blob, size_t* blob_len) {
    std::vector<uint8_t> b = serialize_blob(d);
    if (match_only) {
        uint32_t flags = 1;
        std::memcpy(b.data() + 8 + 16, &flags, 4);  // header.flags; not covered by the body checksum
    }
    void* p = std::malloc(b.size());
    if (!p) return fail(GORP_E_OOM, "out of host memory");
    std::memcpy(p, b.data(), b.size());
    *blob = p;
    *blob_len = b.size();
    return GORP_OK;
}

}  // namespace

// First index i with off[i + 1] < off[i], or -1: the caller's offsets must be non-decreasing. Checked up front (an O(n) scan,
// branch-free inner loop, split over a few threads for batches of millions of lines: 25 M offsets took 20 ms of a 87 ms call
// when scanned by one thread with an early-exit branch).
static int64_t first_decreasing_offset(const int64_t* off, int64_t n_lines) {
    auto scan = [off](int64_t i0, int64_t i1) -> int64_t {
        for (int64_t b = i0; b < i1; b += 4096) {
            const int64_t e = std::min<int64_t>(b + 4096, i1);
            int bad = 0;
            for (int64_t i = b; i < e; ++i) bad |= off[i + 1] < off[i];
            if (bad)
                for (int64_t i = b; i < e; ++i)
                    if (off[i + 1] < off[i]) return i;
        }
        return -1;
    };
    const int n_thr = n_lines >= (1 << 20) ? static_cast<int>(std::min<unsigned>(8, std::max(1u, std::thread::hardware_concurrency()))) : 1;
    if (n_thr == 1) return scan(0, n_lines);
    std::vector<int64_t> first(n_thr, -1);
    std::vector<std::thread> pool;
    for (int t = 0; t < n_thr; ++t)
        pool.emplace_back([&first, &scan, n_lines, n_thr, t] { first[t] = scan(n_lines * t / n_thr, n_lines * (t + 1) / n_thr); });
    for (auto& th : pool) th.join();
    for (int64_t f : first)
        if (f >= 0) return f;
    return -1;
}

extern "C" {

int gorp_abi_version(void) { return GORP_ABI_VERSION; }

const char* gorp_last_error(void) { return g_error.c_str(); }

int gorp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int gorp_compile_definition(const char* grp_utf8, size_t len, void** blob, size_t* blob_len) {
    if (!grp_utf8 || !blob || !blob_len) return fail(GORP_E_ARG, "null argument");
    return guarded([&]() -> int { return export_blob(compile_definition(utf8_to_utf16(grp_utf8, len)), false, blob, blob_len); });
}

int gorp_compile_patterns(const uint16_t* const* patterns, const uint32_t* lens, uint32_t n, void** blob, size_t* blob_len) {
    if (!patterns || !lens || !blob || !blob_len || n == 0) return fail(GORP_E_ARG, "null argument");
    return guarded([&]() -> int {
        CompiledDefinition d;
        std::vector<ustring> pats;
        for (uint32_t i = 0; i < n; ++i) pats.emplace_back(reinterpret_cast<const char16_t*>(patterns[i]), lens[i]);
        d.dfa = compile_patterns(pats);
        for (uint32_t i = 0; i < n; ++i) {
            CompiledExtraction x;
            x.strings.name = utf8_to_utf16(strfmt("#%u", i).c_str(), strfmt("#%u", i).size());
            x.strings.automaton_regex = pats[i];
            d.extractions.push_back(std::move(x));
        }
        return export_blob(d, true, blob, blob_len);
    });
}

void gorp_blob_free(void* blob) { std::free(blob); }

int gorp_blob_get_info(const void* blob, size_t len, gorp_blob_info* out) {
    if (!blob || !out) return fail(GORP_E_ARG, "null argument");
    return guarded([&]() -> int {
        BlobView v;
        view_blob(blob, len, v);
        out->n_states = v.S;
        out->n_classes = v.C;
        out->n_extractions = v.E;
        out->reserved = 0;
        return GORP_OK;
    });
}

int gorp_blob_get_extraction(const void* blob, size_t len, uint32_t index, gorp_extraction_info* out) {
    if (!blob || !out) return fail(GORP_E_ARG, "null argument");
    return guarded([&]() -> int {
        BlobView v;
        view_blob(blob, len, v);
        if (index >= v.E) return fail(GORP_E_ARG, "extraction index out of range");
        locate_extraction(v, index, out, 0, nullptr);
        return GORP_OK;
    });
}

int gorp_blob_get_extractor_name(const void* blob, size_t len, uint32_t extraction, uint32_t k, const uint16_t** name,
                                 uint32_t* name_len) {
    if (!blob || !name || !name_len) return fail(GORP_E_ARG, "null argument");
    return guarded([&]() -> int {
        BlobView v;
        view_blob(blob, len, v);
        if (extraction >= v.E) return fail(GORP_E_ARG, "extraction index out of range");
        gorp_extraction_info info{};
        StrRef s{nullptr, 0};
        locate_extraction(v, extraction, &info, k, &s);
        if (k >= info.n_extractor_names) return fail(GORP_E_ARG, "extractor index out of range");
        *name = s.p;
        *name_len = s.n;
        return GORP_OK;
    });
}

int gorp_blob_get_tables(const void* blob, size_t len, const uint16_t** classmap, const int32_t** transitions,
                         const int32_t** accept_first, const uint32_t** accept_off, const int32_t** accept_list) {
    if (!blob) return fail(GORP_E_ARG, "null argument");
    return guarded([&]() -> int {
        BlobView v;
        view_blob(blob, len, v);
        if (classmap) *classmap = reinterpret_cast<const uint16_t*>(v.base + v.classmap);
        if (transitions) *transitions = reinterpret_cast<const int32_t*>(v.base + v.trans);
        if (accept_first) *accept_first = reinterpret_cast<const int32_t*>(v.base + v.acc_first);
        if (accept_off) *accept_off = reinterpret_cast<const uint32_t*>(v.base + v.acc_off);
        if (accept_list) *accept_list = reinterpret_cast<const int32_t*>(v.base + v.acc_list);
        return GORP_OK;
    });
}

int gorp_engine_create(const void* blob, size_t len, const int* devices, int n_devices, gorp_engine** out) {
    if (!blob || !out) return fail(GORP_E_ARG, "null argument");
    *out = nullptr;
    return guarded([&]() -> int {
        auto eng = std::make_unique<gorp_engine>();
        eng->def = parse_blob(blob, len);
        uint32_t flags;
        std::memcpy(&flags, static_cast<const uint8_t*>(blob) + 8 + 16, 4);
        eng->match_only = (flags & 1u) != 0;
        DeviceModel model;
        FusedAutomaton fused;
        TailSet tailset;
        if (eng->match_only) {
            model.dfa = compact_tables(eng->def.dfa);
            model.n_groups.assign(eng->def.extractions.size(), 0);
        } else {
            model = build_device_model(eng->def);
            fused = build_fused(model);
            finalize_device_model(model, fused);
            if (!std::getenv("GORP_NO_TAILS")) tailset = build_tails(eng->def, model);
        }
        int avail = 0;
        if (cudaGetDeviceCount(&avail) != cudaSuccess || avail == 0) {
            cudaGetLastError();
            return fail(GORP_E_CUDA, "no CUDA device available (libgorpcuda has no CPU fallback)");
        }
        std::vector<int> devs;
        if (devices && n_devices > 0) devs.assign(devices, devices + n_devices);
        else devs.push_back(0);
        for (int d : devs) {
            if (d < 0 || d >= avail) return fail(GORP_E_ARG, strfmt("device %d out of range (have %d)", d, avail));
            auto ctx = std::make_unique<DeviceCtx>();
            ctx->device = d;
            build_device(*ctx, model, fused, tailset, eng->def.dfa, eng->match_only);
            eng->devs.push_back(std::move(ctx));
        }
        *out = eng.release();
        return GORP_OK;
    });
}

void gorp_engine_destroy(gorp_engine* e) { delete e; }

int gorp_extract_lines(gorp_engine* e, const uint16_t* text, const int64_t* off, int64_t n_lines, gorp_result* out) {
    if (!e || !out || !off || n_lines < 0) return fail(GORP_E_ARG, "bad argument");
    // the offsets come from the caller: anything that is not a non-decreasing sequence starting at >= 0 would send the
    // kernels outside the staged text
    if (off[0] < 0) return fail(GORP_E_ARG, "offsets must start at >= 0");
    if (const int64_t i = first_decreasing_offset(off, n_lines); i >= 0)
        return fail(GORP_E_ARG, strfmt("offsets must be non-decreasing (line %lld)", static_cast<long long>(i)));
    return extract_host(e, text, nullptr, n_lines > 0 ? off[n_lines] : 0, off, n_lines, out);
}

int gorp_extract_text(gorp_engine* e, const uint16_t* text, int64_t n_units, gorp_result* out) {
    return extract_host(e, text, nullptr, n_units, nullptr, 0, out);
}

int gorp_extract_text_latin1(gorp_engine* e, const uint8_t* text, int64_t n_bytes, gorp_result* out) {
    return extract_host(e, nullptr, text, n_bytes, nullptr, 0, out);
}

int gorp_extract_text_utf8(gorp_engine* e, const uint8_t* text, int64_t n_bytes, gorp_result* out) {
    return extract_host(e, nullptr, text, n_bytes, nullptr, 0, out, true);
}

int gorp_extract_text_utf8_bytes(gorp_engine* e, const uint8_t* text, int64_t n_bytes, gorp_result* out) {
    return extract_host(e, nullptr, text, n_bytes, nullptr, 0, out, true, true);
}

static int extract_lines_utf8(gorp_engine* e, const uint8_t* text, const int64_t* off, int64_t n_lines, gorp_result* out,
                              gorp_device_tables* tables) {
    if (!e || !out || !off || n_lines < 0) return fail(GORP_E_ARG, "bad argument");
    if (off[0] < 0) return fail(GORP_E_ARG, "offsets must start at >= 0");
    if (const int64_t i = first_decreasing_offset(off, n_lines); i >= 0)
        return fail(GORP_E_ARG, strfmt("offsets must be non-decreasing (line %lld)", static_cast<long long>(i)));
    return extract_host(e, nullptr, text, n_lines > 0 ? off[n_lines] : 0, off, n_lines, out, true, true, tables);
}

int gorp_extract_lines_utf8(gorp_engine* e, const uint8_t* text, const int64_t* off, int64_t n_lines, gorp_result* out) {
    return extract_lines_utf8(e, text, off, n_lines, out, nullptr);
}

int gorp_extract_text_utf8_tables(gorp_engine* e, const uint8_t* text, int64_t n_bytes, gorp_result* out, gorp_device_tables* tables) {
    if (!tables) return fail(GORP_E_ARG, "bad argument");
    return extract_host(e, nullptr, text, n_bytes, nullptr, 0, out, true, true, tables);
}

int gorp_extract_lines_utf8_tables(gorp_engine* e, const uint8_t* text, const int64_t* off, int64_t n_lines, gorp_result* out,
                                   gorp_device_tables* tables) {
    if (!tables) return fail(GORP_E_ARG, "bad argument");
    return extract_lines_utf8(e, text, off, n_lines, out, tables);
}

int gorp_match_all_lines(gorp_engine* e, const uint16_t* text, const int64_t* off, int64_t n_lines, gorp_match_result* out) {
    if (!e || !out || !off || n_lines < 0 || e->devs.empty()) return fail(GORP_E_ARG, "bad argument");
    if (off[0] < 0) return fail(GORP_E_ARG, "offsets must start at >= 0");
    if (const int64_t i = first_decreasing_offset(off, n_lines); i >= 0)
        return fail(GORP_E_ARG, strfmt("offsets must be non-decreasing (line %lld)", static_cast<long long>(i)));
    if (!text && n_lines > 0 && off[n_lines] > off[0]) return fail(GORP_E_ARG, "null text");
    return guarded([&]() -> int {
        DeviceCtx& c = *e->devs[0];
        CtxLock lock(c);
        DeviceGuard restore_device;
        CK(cudaSetDevice(c.device));
        CK(cudaStreamWaitEvent(c.stream, c.ev_done, 0));
        Launch L{c.stream, c.sm_count};
        const size_t nl = static_cast<size_t>(n_lines);
        const int64_t u0 = n_lines ? off[0] : 0, u1 = n_lines ? off[n_lines] : 0;
        c.textbuf[0].reserve(static_cast<size_t>(u1 - u0 + 64) * 2);
        c.offbuf[0].reserve((nl + 1) * 8);
        c.ma_state.reserve((nl + 1) * 4);
        c.ma_count.reserve((nl + 1) * 4);
        c.ma_off.reserve((nl + 2) * 8);
        c.scan_scratch.reserve((nl / 4096 + 8) * 8);
        std::unique_ptr<HostResult> hr = std::make_unique<HostResult>();
        hr->numa_node = c.numa_node;
        hr->reserve(1, (nl + 2) * 8);
        int64_t total = 0;
        if (n_lines > 0) {
            if (u1 > u0) CK(cudaMemcpyAsync(c.textbuf[0].p, text + u0, static_cast<size_t>(u1 - u0) * 2, cudaMemcpyHostToDevice, c.stream));
            CK(cudaMemcpyAsync(c.offbuf[0].p, off, (nl + 1) * 8, cudaMemcpyHostToDevice, c.stream));
            // text[i] lives at textbuf + (i - u0)
            k_matchall_walk(L, c.matchall, c.textbuf[0].as<uint16_t>() - u0, c.offbuf[0].as<int64_t>(), n_lines, c.ma_state.as<int32_t>(),
                            c.ma_count.as<uint32_t>());
            scan_u32_to_i64(L, c.ma_count.as<uint32_t>(), n_lines, c.ma_off.as<int64_t>(), c.scan_scratch.as<int64_t>());
            CK(cudaMemcpyAsync(&total, c.ma_off.as<int64_t>() + n_lines, 8, cudaMemcpyDeviceToHost, c.stream));
            CK(cudaStreamSynchronize(c.stream));
            c.ma_out.reserve(static_cast<size_t>(total + 1) * 4);
            k_matchall_fill(L, c.matchall, c.ma_state.as<int32_t>(), c.ma_off.as<int64_t>(), n_lines, c.ma_out.as<int32_t>());
            c.launches += 5;
            hr->reserve(0, static_cast<size_t>(total + 1) * 4);
            CK(cudaMemcpyAsync(hr->p[1], c.ma_off.p, (nl + 1) * 8, cudaMemcpyDeviceToHost, c.stream));
            if (total) CK(cudaMemcpyAsync(hr->p[0], c.ma_out.p, static_cast<size_t>(total) * 4, cudaMemcpyDeviceToHost, c.stream));
            CK(cudaStreamSynchronize(c.stream));
        } else {
            hr->reserve(0, 4);
            static_cast<int64_t*>(hr->p[1])[0] = 0;
        }
        CK(cudaEventRecord(c.ev_done, c.stream));
        out->n_lines = n_lines;
        out->accept_off = static_cast<const int64_t*>(hr->p[1]);
        out->accept = static_cast<const int32_t*>(hr->p[0]);
        out->owner = hr.release();
        return GORP_OK;
    });
}

void gorp_match_result_release(gorp_engine* e, gorp_match_result* r) {
    (void)e;
    if (!r || !r->owner) return;
    delete static_cast<HostResult*>(r->owner);
    r->owner = nullptr;
}

void gorp_result_release(gorp_engine* e, gorp_result* r) {
    if (!r || !r->owner) return;
    std::unique_ptr<HostResult> hr(static_cast<HostResult*>(r->owner));
    r->owner = nullptr;
    if (e) {
        std::lock_guard<std::mutex> pl(e->pool_mu);
        if (e->pool.size() < 4) e->pool.push_back(std::move(hr));
    }
}

int gorp_extract_text_device(gorp_engine* e, int dev_index, const uint16_t* d_text, int64_t n_units, void* stream, int flags,
                             gorp_device_result* out) {
    if (!e || dev_index < 0 || dev_index >= static_cast<int>(e->devs.size()) || n_units < 0 || (reinterpret_cast<uintptr_t>(d_text) & 15))
        return fail(GORP_E_ARG, "bad argument (d_text must be 16-byte aligned)");
    return guarded([&]() -> int {
        DeviceCtx& c = *e->devs[dev_index];
        CtxLock lock(c);
        DeviceGuard restore_device;
        CK(cudaSetDevice(c.device));
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        CK(cudaStreamWaitEvent(st, c.ev_done, 0));  // the previous call on this context (any stream) used the same scratch
        Timer tm(c, st, (flags & GORP_FLAG_TIME_KERNELS) != 0);
        run_pipeline(c, d_text, n_units, nullptr, 0, st, tm, &c.last);
        if (out) *out = c.last;
        CK(cudaEventRecord(c.ev_done, st));
        c.last_unit_bytes = 2;
        c.last_text = d_text;
        if (flags & GORP_FLAG_SYNC) CK(cudaStreamSynchronize(st));
        return GORP_OK;
    });
}

int gorp_extract_lines_device(gorp_engine* e, int dev_index, const uint16_t* d_text, const int64_t* d_off, int64_t n_lines,
                              void* stream, int flags, gorp_device_result* out) {
    if (!e || dev_index < 0 || dev_index >= static_cast<int>(e->devs.size()) || !d_off || n_lines < 0 ||
        (reinterpret_cast<uintptr_t>(d_text) & 15))
        return fail(GORP_E_ARG, "bad argument (d_text must be 16-byte aligned)");
    return guarded([&]() -> int {
        DeviceCtx& c = *e->devs[dev_index];
        CtxLock lock(c);
        DeviceGuard restore_device;
        CK(cudaSetDevice(c.device));
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        CK(cudaStreamWaitEvent(st, c.ev_done, 0));  // the previous call on this context (any stream) used the same scratch
        int64_t n_units = 0;  // the extent of the text = the last offset (the block walkers must not read beyond it)
        if (n_lines > 0 && c.tails.enabled) {
            CK(cudaMemcpyAsync(&n_units, d_off + n_lines, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        Timer tm(c, st, (flags & GORP_FLAG_TIME_KERNELS) != 0);
        run_pipeline(c, d_text, n_units, d_off, n_lines, st, tm, &c.last);
        if (out) *out = c.last;
        CK(cudaEventRecord(c.ev_done, st));
        c.last_unit_bytes = 2;
        c.last_text = d_text;
        if (flags & GORP_FLAG_SYNC) CK(cudaStreamSynchronize(st));
        return GORP_OK;
    });
}

int gorp_extract_text_utf8_device(gorp_engine* e, int dev_index, const uint8_t* d_text, int64_t n_bytes, void* stream, int flags,
                                  gorp_device_result* out) {
    if (!e || dev_index < 0 || dev_index >= static_cast<int>(e->devs.size()) || n_bytes < 0 || (reinterpret_cast<uintptr_t>(d_text) & 15))
        return fail(GORP_E_ARG, "bad argument (d_text must be 16-byte aligned)");
    return guarded([&]() -> int {
        DeviceCtx& c = *e->devs[dev_index];
        CtxLock lock(c);
        DeviceGuard restore_device;
        CK(cudaSetDevice(c.device));
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        CK(cudaStreamWaitEvent(st, c.ev_done, 0));  // the previous call on this context (any stream) used the same scratch
        Launch L{st, c.sm_count};
        Timer tm(c, st, (flags & GORP_FLAG_TIME_KERNELS) != 0);
        // round trip 1: {decoded total, first malformed byte, last byte}; round trip 2: the newline count (run_pipeline)
        c.textbuf[0].reserve(static_cast<size_t>(n_bytes + 64) * 2);
        uint16_t* text = c.textbuf[0].as<uint16_t>();
        uint8_t last = 0x0A;
        const int64_t n_units = utf8_text_decode(c, L, tm, d_text, n_bytes, 0, text, &last);
        gorp_device_result dr{};
        run_pipeline(c, text, n_units, nullptr, 0, st, tm, &dr);
        const uint32_t stride = static_cast<uint32_t>(dr.span_stride);
        reserve_byte_rows(c, dr.n_lines, stride, true);
        utf8_text_rows(c, L, tm, d_text, n_bytes, last == 0x0A, dr, 0, stride, c.acc_off.as<int64_t>(), c.acc_spans.as<int32_t>());
        CK(cudaGetLastError());
        dr.d_line_off = c.acc_off.as<int64_t>();
        dr.d_spans = c.acc_spans.as<int32_t>();
        if (out) *out = dr;
        CK(cudaEventRecord(c.ev_done, st));
        c.last = dr;
        c.last_unit_bytes = 1;
        c.last_text = d_text;
        if (flags & GORP_FLAG_SYNC) CK(cudaStreamSynchronize(st));
        return GORP_OK;
    });
}

int gorp_extract_lines_utf8_device(gorp_engine* e, int dev_index, const uint8_t* d_text, const int64_t* d_off, int64_t n_lines, void* stream,
                                   int flags, gorp_device_result* out) {
    if (!e || dev_index < 0 || dev_index >= static_cast<int>(e->devs.size()) || !d_off || n_lines < 0 ||
        (reinterpret_cast<uintptr_t>(d_text) & 15))
        return fail(GORP_E_ARG, "bad argument (d_text must be 16-byte aligned)");
    return guarded([&]() -> int {
        DeviceCtx& c = *e->devs[dev_index];
        CtxLock lock(c);
        DeviceGuard restore_device;
        CK(cudaSetDevice(c.device));
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        CK(cudaStreamWaitEvent(st, c.ev_done, 0));  // the previous call on this context (any stream) used the same scratch
        Launch L{st, c.sm_count};
        Timer tm(c, st, (flags & GORP_FLAG_TIME_KERNELS) != 0);
        // round trip 1: d_off[0] and d_off[n_lines] size the copy and the decode buffer
        int64_t ends[2] = {0, 0};
        CK(cudaMemcpyAsync(&ends[0], d_off, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&ends[1], d_off + n_lines, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (ends[0] < 0) throw ArgError("offsets must start at >= 0");
        // (d_off[n] < d_off[0]: some offset decreases, which the order check of utf8_lines_decode reports; nothing is read)
        const int64_t at = ends[0], n_bytes = std::max<int64_t>(ends[1] - at, 0);
        // the strings' bytes are copied to the 16-byte aligned staging buffer, so every kernel sees the layout of a staged
        // host piece whatever the alignment of d_off[0], and no byte outside [d_off[0], d_off[n]) is read
        c.bytebuf[0].reserve(static_cast<size_t>(n_bytes) + 64);
        c.textbuf[0].reserve(static_cast<size_t>(n_bytes + kTextPad + 64) * 2);
        c.unit_off.reserve(static_cast<size_t>(n_lines + 1) * 8);
        c.slice_units.reserve(static_cast<size_t>(n_bytes / 16 + 1) * 2);
        const uint8_t* bytes = c.bytebuf[0].as<uint8_t>();
        if (n_bytes) CK(cudaMemcpyAsync(c.bytebuf[0].p, d_text + at, static_cast<size_t>(n_bytes), cudaMemcpyDeviceToDevice, st));
        tm.mark("utf8_copy", 0);
        // round trip 2: {decoded total, first malformed byte, first decreasing offset}
        uint16_t* text = c.textbuf[0].as<uint16_t>() + kTextPad;  // (device address - unit index) a multiple of 32 bytes
        const int64_t n_units = utf8_lines_decode(c, L, tm, bytes, n_bytes, at, d_off, n_lines, text, true);
        gorp_device_result dr{};
        run_pipeline(c, text, n_units, c.unit_off.as<int64_t>(), n_lines, st, tm, &dr);
        const uint32_t stride = static_cast<uint32_t>(dr.span_stride);
        reserve_byte_rows(c, n_lines, stride, false);
        utf8_lines_rows(L, tm, bytes, at, d_off, dr, stride, nullptr, c.acc_spans.as<int32_t>());  // (d_line_off is d_off itself)
        CK(cudaGetLastError());
        dr.d_line_off = d_off;
        dr.d_spans = c.acc_spans.as<int32_t>();
        if (out) *out = dr;
        CK(cudaEventRecord(c.ev_done, st));
        c.last = dr;
        c.last_unit_bytes = 1;
        c.last_text = d_text;
        if (flags & GORP_FLAG_SYNC) CK(cudaStreamSynchronize(st));
        return GORP_OK;
    });
}

int gorp_extract_tables_device(gorp_engine* e, int dev_index, void* stream, int flags, gorp_device_tables* out) {
    if (!e || !out || dev_index < 0 || dev_index >= static_cast<int>(e->devs.size())) return fail(GORP_E_ARG, "bad argument");
    return guarded([&]() -> int {
        DeviceCtx& c = *e->devs[dev_index];
        std::lock_guard<std::mutex> lock(c.mu);  // (not CtxLock: the tables leave the result they read as it is)
        if (!c.last_unit_bytes)
            throw ArgError("no device-resident result to make tables of: the last call on this engine and device must be a successful "
                           "gorp_extract_*_device call");
        DeviceGuard restore_device;
        CK(cudaSetDevice(c.device));
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        CK(cudaStreamWaitEvent(st, c.ev_done, 0));  // the previous call on this context (any stream) used the same scratch
        Timer tm(c, st, (flags & GORP_FLAG_TIME_KERNELS) != 0);
        TablesBuilt b;
        build_tables(e, c, st, tm, c.last, c.last_text, c.last_unit_bytes, b);
        c.tb_desc.reset(c.n_ext, b.n_cols);
        for (uint32_t t = 0; t < c.n_ext; ++t) {
            const TableLayout& x = b.lay[t];
            for (int64_t k = 0; k < x.n_cols; ++k) {
                const int64_t col = x.col_base + k;
                c.tb_desc.offsets[col] = c.tb_offs.as<int64_t>() + x.off_base + k * x.seg;
                c.tb_desc.data[col] = c.tb_data.as<uint8_t>() + b.col_info[2 * col + 1];
                c.tb_desc.valid[col] = reinterpret_cast<const uint8_t*>(c.tb_valid.as<uint32_t>() + x.valid_base + k * x.vwords);
                c.tb_desc.nulls[col] = b.stats[2 * col + 1];
            }
            c.tb_desc.set_table(t, x.n_rows, c.tb_rows.as<int64_t>() + x.row_base, x.col_base, x.n_cols);
        }
        c.tb_desc.describe(out, c.last_unit_bytes);
        CK(cudaEventRecord(c.ev_done, st));
        if (flags & GORP_FLAG_SYNC) CK(cudaStreamSynchronize(st));
        return GORP_OK;
    });
}

int gorp_kernel_times(gorp_engine* e, int dev_index, const char** names, double* total_ms, int cap, int* n, int64_t* calls,
                       int64_t* launches, int reset) {
    if (!e || dev_index < 0 || dev_index >= static_cast<int>(e->devs.size()) || !n) return fail(GORP_E_ARG, "bad argument");
    DeviceCtx& c = *e->devs[dev_index];
    std::lock_guard<std::mutex> lock(c.mu);
    DeviceGuard restore_device;
    cudaSetDevice(c.device);
    collect_times(c);
    int k = std::min(cap, c.acc_n);
    for (int i = 0; i < k; ++i) {
        if (names) names[i] = c.ev_name[i];
        if (total_ms) total_ms[i] = c.acc_ms[i];
    }
    *n = k;
    if (calls) *calls = c.acc_calls;
    if (launches) *launches = c.launches;
    if (reset) {
        for (auto& v : c.acc_ms) v = 0;
        c.acc_calls = 0;
        c.acc_n = 0;
        c.launches = 0;
    }
    return GORP_OK;
}

}  // extern "C"
