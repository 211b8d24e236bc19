// Device-side data layout and kernel entry points of libgorpcuda (sm_100a).
//
// Reference functions each kernel stands in for (gorp-core/src/main/java/com/salesforce/gorp/):
//   K1 newline index    — no counterpart (callers of Gorp.extract pre-split lines, Gorp.java:145)
//   K2 dfa_scan         — PolyMatcher.match + Automata.step/accept (autom/PolyMatcher.java:123-133,
//                         autom/Automata.java:133-139) and the first-index dispatch of Gorp.java:166-167
//   K4 tdfa_capture     — JDKRegexpCookedExtraction.match/_constructMatch (jdkre/JDKRegexpCookedExtraction.java:36-59)
//   K3 histogram, fixed-stride result rows — result assembly of model/CookedExtraction.java:54-57
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gorp {

constexpr int kMaxTdfaRegs = 32;   // run-time register file per line (tag registers of the capture automaton)
constexpr int kMaxTdfaRegsBig = 256;  // ... of the variant for capture automata with more registers (host limit: 250)
constexpr int kCapFastThreads = 512;  // CTA size of the fast capture tier (register offsets in the capture image are
                                      // pre-multiplied by kCapFastThreads * 4)

struct DfaDev {                    // combined multi-regex DFA, compacted (host/automata.hpp: CompactDfa)
    const uint16_t* cls;           // [65536] unit -> class
    const void* trans;             // [(S+1)*(C+1)] premultiplied next-row offset (next*(C+1)); u16 entries, or u32
                                   // when `wide`. Row S = dead (absorbing); column C = identity (self-loop).
    const int32_t* accept_first;   // [S+1], entry S = -1
    uint32_t n_states, n_classes;  // S, C (without the dead row / identity column)
    uint32_t wide;
};

struct ExtDev {                    // per-extraction capture automaton (host/capture.hpp: Tdfa)
    uint32_t n_states;             // S; row S of the table = dead (absorbing, not accepting)
    uint32_t trans_off;            // into tdfa_trans: [(S+1) * (n_classes+1)], last column = identity
    uint32_t opoff_off;            // into tdfa_op_off
    uint32_t ops_off;              // into tdfa_ops
    uint32_t fin_off;              // into tdfa_fin
    uint32_t acc_off;              // into tdfa_accepting
    uint32_t n_slots;              // 2 * groups
};

struct CapDev {
    const uint16_t* cls;           // [65536] unit -> symbol class of the capture automata
    uint32_t n_classes, pair_hi_class;
    const ExtDev* ext;             // [E]
    const uint32_t* tdfa_trans;    // next(16) | oplist(16)
    const uint32_t* tdfa_op_off;
    const uint16_t* tdfa_ops;      // (dst << 8) | src, src 0xFF = position
    const uint8_t* tdfa_fin;
    const uint8_t* tdfa_accepting;
    uint32_t n_ext;
    uint32_t match_only;
    uint32_t max_regs;             // widest register file among the extractions
};

// K2 fast tier ("T0"): combined DFA as directly ASCII-indexed rows in shared memory, text form only.
// Row r = 128 u32 entries (512 B) holding the NEXT ROW; the kernel rewrites them into absolute shared-memory
// addresses, so one step is  addr = state + unit*4 ; state = LDS[addr].  Rows:
//   [0, S)               DFA states (0 = start); column '\n' leads to FIN(accept_first(state))
//   [skip_base, +7)      SKIP_1..SKIP_7: swallow the units that precede the line inside its first 16-byte chunk
//   [fin_base, +1+E)     FIN(-1) (= dead, no match), FIN(0..E-1): absorbing; reached at the line's '\n'
// A chunk that holds any unit >= 0x80 takes the slow per-unit path through the class map (global memory).
struct DfaDirectDev {
    const uint32_t* rows;          // [n_rows * 128] next row index
    uint32_t n_rows, n_states, skip_base, fin_base;
    const uint16_t* cls;           // [65536] slow path: unit -> class
    const int32_t* trans_plain;    // [S*C]   slow path: next state or -1
    const int32_t* accept_first;   // [S]
    uint32_t n_classes;
    uint32_t enabled;
};

// K4 fast tier: per-extraction capture automaton as class-indexed rows in shared memory, text form only.
// Row layout per extraction (row = n_cols u32 entries): [0,S) states, [S,S+7) SKIP_1..7, S+7 DEAD, S+8 SLOW (trap),
// S+9+s FRZ(s) (reached at the line's '\n' from state s; absorbing). Entry: bits 2..15 next row byte offset (relative
// to the extraction's table), bits 16..31 byte offset of the tag register to set to the current position (or of the
// per-thread dummy register). Transitions that need more than "one register := position" lead to SLOW and the chunk
// is replayed through the general tables. Tag registers live in shared memory: reg r of thread t at r*blockDim*4 + t*4.
struct FastExtDev {
    uint32_t tab_off;      // byte offset of this extraction's table inside the shared-memory image
    uint32_t row_bytes;    // n_cols * 4
    uint32_t n_states;
    uint32_t dead_off;     // (S+7) * row_bytes ; everything >= dead_off stops the walk
    uint32_t slow_off;     // (S+8) * row_bytes
    uint32_t frz_off;      // (S+9) * row_bytes
};

struct TdfaFastDev {
    const uint32_t* image;       // [image_words] = cls128 (pre-scaled class*4) followed by all tables
    uint32_t image_words;
    uint32_t n_regs;             // tag registers incl. scratch; register n_regs = dummy, n_regs + 1 = LEN (the line
                                 // length, stored by the '\n' transition); n_regs + 2 registers per thread
    const FastExtDev* ext;       // [E]
    uint32_t enabled;
};

struct Launch {
    cudaStream_t stream;
    int sm_count;
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is per-function, per-device state shared by every engine of the process:
// it is always set to the same value (everything the device allows), so launches of engines with different table
// sizes cannot invalidate each other's setting; only the launch's own dynamic shared-memory argument varies.
template <class Kernel>
inline void allow_max_dynamic_smem(Kernel kernel) {
    cudaFuncAttributes a{};
    int dev = 0, optin = 0;
    if (cudaFuncGetAttributes(&a, kernel) != cudaSuccess || cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - static_cast<int>(a.sharedSizeBytes));
}

// K1: '\n' index over UTF-16 text. tile_counts/tile_base sized ceil(n_units / kNlTile).
constexpr int kNlTile = 8192;
void k1_count_newlines(const Launch&, const uint16_t* text, int64_t n_units, uint32_t* tile_counts);
void k1_scatter_newlines(const Launch&, const uint16_t* text, int64_t n_units, const int64_t* tile_base,
                         int64_t* line_off /* entries 1.. */);
// same pair with the '\n' masks (one u32 per 32 units, ceil(n_units / kNlTile) * 256 words) as a side product of the
// count pass: the scatter pass then reads the masks instead of the text (one HBM pass over the text instead of two)
void k1_count_newlines_masks(const Launch&, const uint16_t* text, int64_t n_units, uint32_t* tile_counts, uint32_t* masks);
void k1_scatter_masks(const Launch&, const uint32_t* masks, int64_t n_units, const int64_t* tile_base, int64_t* line_off);
void k1_finish(const Launch&, const uint16_t* text, int64_t n_units, const int64_t* total_newlines, int64_t* line_off,
               int64_t* n_lines_out);

// exclusive scan: out[i] = sum_{j<i} in[j], out[n] = total (int64). scratch >= ceil(n/4096)+1 int64.
void scan_u32_to_i64(const Launch&, const uint32_t* in, int64_t n, int64_t* out, int64_t* scratch);

// K2: combined DFA, one line per thread. Writes ext_id (>=0 | -1).
void k2_dfa_scan(const Launch&, const DfaDev&, const uint16_t* text, const int64_t* line_off, int sep, int64_t n_lines,
                 int32_t* ext_id);

// K2 fast tier: lines [0, n_lines) must each be terminated by '\n' in the text (the caller excludes a final
// unterminated line and runs it through k2_dfa_scan).
void k2_dfa_direct(const Launch&, const DfaDirectDev&, const uint16_t* text, const int64_t* line_off, int64_t n_lines,
                   int32_t* ext_id);

// K4: capture automaton over the matched lines. Writes the result row spans[i*span_stride ..]: 2*groups entries, the
// rest of the row (and the whole row of a MISS / capture-failed line) is -1; capture failure => ext_id = -2-e.
// `skip_tails` (optional): only the lines whose extraction has no tail automaton are walked (the tail walk owns the others and
// the bucket pass has filled the MISS rows); `hist` (optional): a capture failure moves the line's count (K3 ran before).
struct TailExt;
void k4_tdfa_capture(const Launch&, const CapDev&, const uint16_t* text, const int64_t* line_off, int sep, int64_t n_lines,
                     uint32_t span_stride, int32_t* ext_id, int32_t* spans, const TailExt* skip_tails = nullptr,
                     unsigned long long* hist = nullptr);

// K4 fast tier: lines [0, n_lines) are '\n'-terminated in the text.
void k4_tdfa_fast(const Launch&, const TdfaFastDev&, const CapDev&, const uint16_t* text, int64_t n_units,
                  const int64_t* line_off, int64_t n_lines, uint32_t span_stride, int32_t* ext_id, int32_t* spans);

// K2b: combined-DFA walk over an existing line index (K1, or the caller's offsets), lanes pull lines dynamically — see
// kernels/dfawalk.cu. Writes ext_id (>= 0 | -1; the candidate when `a` is the early-exit table and the tail walk follows).
// Text form: every line must be terminated by '\n' in the text or end at n_units.
struct DfaWalkDev {
    const uint16_t* table;       // [n_rows * K] next row (global copy, padded to 16 bytes; copied to shared memory
                                 // when it fits). Rows: [0,S) states, S = DEADSCAN, S+1..S+15 = SKIP_1..15,
                                 // fin_base = S+16: FIN(-1), then FIN(0..E-1). Column K-1 = '\n'.
    uint32_t n_rows, K;
    uint32_t n_states, fin_base;
    const uint16_t* cls128;      // [128] ASCII unit -> byte offset of its column inside a row (2 * column)
    const uint16_t* xcls;        // [65536] unit -> column (units >= 0x80)
    uint32_t enabled;
};
constexpr uint32_t kLineItemLines = 1024;
struct LineWalkParams {
    const uint16_t* text;
    int64_t n_units;
    const int64_t* line_off;
    int64_t n_lines;
    DfaWalkDev a;
    int32_t* ext_id;
    unsigned int* item_ticket;   // zeroed by the caller
    uint32_t flags;              // GORP_WALK_FLAGS (diagnostics): 1 = text loads L2 evict-first
    uint32_t lines_form;         // 1: List<String> form — line i = [line_off[i], line_off[i+1]), a '\n' is content
};
bool k2b_linewalk_plan(const DfaWalkDev&, uint32_t* threads, bool* in_smem);
void k2b_linewalk_scan(const Launch&, const LineWalkParams&, uint32_t threads, bool in_smem);

// K4b: capture half of the text form, bucketed by extraction — see kernels/capwalk.cu.
constexpr uint32_t kCapItemLines = 4096;   // lines per work item (one CTA walks one item)
constexpr uint32_t kCapMaxBuckets = 4096;  // extractions the bucket kernels hold in shared memory
constexpr int kCapWalkThreads = 256;
struct CapItem {
    uint32_t ext, begin, end;    // entries [begin, end) of `perm` are lines of extraction `ext`
};
struct CapImgExt {               // per-extraction table inside the image (byte offsets)
    uint32_t tab_off;            // of the table inside the image
    uint32_t row_bytes;          // K * 4
    uint32_t n_states;
    uint32_t dead_off;           // (S+15) * row_bytes ; everything >= dead_off ends the walk of a line
    uint32_t slow_off;           // (S+16) * row_bytes
    uint32_t frz_off;            // (S+17) * row_bytes
};
struct CapImgDev {
    const uint32_t* image;       // all tables
    const uint32_t* cls128;      // [128] ASCII unit -> class * 4 ('\n' -> the last column)
    const CapImgExt* ext;        // [E]
    uint32_t n_regs;             // widest register file; slot n_regs = the per-thread dummy
    uint32_t smem_table_bytes;   // shared memory set aside for the table of the extraction a CTA is working on
    uint32_t enabled;
};
struct CapWalkParams {
    const uint16_t* text;
    int64_t n_units;
    const int64_t* line_off;
    const uint32_t* perm;        // line ids grouped by extraction
    const CapItem* items;
    const uint32_t* n_items;
    uint32_t* item_ticket;
    CapImgDev img;
    CapDev cap;                  // general tables (slow path, final states)
    const struct TailExt* skip_tails;  // extractions whose items the tail walk (kernels/tailwalk.cu) takes, or null
    uint32_t span_stride;
    uint32_t smem_table_bytes;   // = img.smem_table_bytes, or 0 to read every table through L1/L2 (GORP_CAP_FLAGS=2)
    uint32_t flags;              // GORP_WALK_FLAGS (diagnostics): 1 = text loads L2 evict-first
    int32_t* ext_id;
    int32_t* spans;
    unsigned long long* hist;    // [E+2]: a capture failure moves one count from bin e to bin E+1
};
// hist (K3 layout) -> bucket_base[E+1], cursor[E], items (<= n_lines / kCapItemLines + E), perm; MISS rows := -1
struct LineRec;
struct TailExt;
void k4b_bucket(const Launch&, const int32_t* ext_id, int64_t n_lines, uint32_t n_ext, const unsigned long long* hist,
                uint32_t* bucket_base, uint32_t* cursor, uint32_t* perm, CapItem* items, uint32_t* n_items, uint32_t* item_ticket,
                int32_t* spans, uint32_t span_stride, const int64_t* line_off = nullptr, LineRec* recs = nullptr, int sep = 1,
                const TailExt* tails = nullptr,  // tails (with recs): extractions whose lines only need a record, no `perm` entry
                uint32_t item_lines = kCapItemLines, bool interleave = false);  // work items: size, bucket by bucket / by relative position
size_t capwalk_smem_bytes(const CapImgDev&);
void k4b_capwalk(const Launch&, const CapWalkParams&);

// K4c: tail walk — the capture half for extractions that have a tail automaton (host/tails.hpp, host/walktables.hpp:
// TailImage) — see kernels/tailwalk.cu. Decides MISS / MATCH / CAPTURE_FAIL of candidate lines and writes their rows.
constexpr uint32_t kTailMaxLen = 65000;   // lines at least this long take the 32-bit one-thread-per-line kernel
struct TailExt {                 // mirrors host/walktables.hpp: TailImageExt
    uint32_t tab_off;            // byte offset of the table inside the image (16-byte aligned)
    uint32_t n_states, fin_base, n_outcomes;
    uint32_t res_off, oext_off, init_off, n_init, n_slots, available;
};
struct TailDev {
    const uint16_t* image;       // all tables: rows of `width` u16 entries (next row << 6) | op slot
    const TailExt* ext;          // [E]
    const uint32_t* res;         // [n_outcomes * span_stride] per extraction: group boundary recipes
    const int32_t* oext;         // outcome -> ext code (-1 | e | -2-e)
    const uint8_t* init_slots;
    const uint16_t* xcol;        // [65536] unit -> column
    const uint16_t* pair_col;    // [width]
    uint32_t width, row_bytes, span_stride;
    uint32_t max_table_bytes, max_slots, max_res, max_outcomes;  // shared-memory sizing (the largest tail)
    uint32_t nl_data_col;        // column of a '\n' that is line content (List<String> form)
    uint32_t n_without;          // extractions without a tail (their items stay with the bucketed capture walk)
    uint32_t enabled;
};
struct LineRec {                 // what the tail walk needs to start a line, in one 16-byte load (written by the bucket pass)
    int64_t start;               // unit offset of the line
    uint32_t line, len;          // line id; length in units (without the '\n')
};
struct TailWalkParams {
    const uint16_t* text;
    int64_t n_units;
    const int64_t* line_off;
    const LineRec* recs;         // [n_lines] parallel to perm: the lines grouped by (candidate) extraction
    const uint32_t* perm;        // line ids grouped by (candidate) extraction
    const CapItem* items;
    const uint32_t* n_items;
    uint32_t* item_ticket;       // zeroed by the caller
    TailDev t;
    uint32_t n_ext;
    uint32_t round_iters;        // walk iterations (16 units each) between two service points
    uint32_t lines_form;         // 1: List<String> form — lines end where their record says, a '\n' is content
    uint32_t flags;              // GORP_TAIL_FLAGS (diagnostics): 1 = L2 bulk prefetch of the next line, 2 / 4 = text loads ask
                                 // L2 for the 128 / 256-byte neighbourhood, 8 = no just-in-time L2 prefetch four blocks ahead
    int32_t* ext_id;
    int32_t* spans;
    unsigned long long* hist;    // [E+2]: a candidate that ends as MISS / CAPTURE_FAIL moves its count
    uint32_t* long_lines;        // [long_cap] lines handed to the 32-bit kernel
    uint32_t* n_long;            // zeroed by the caller
    uint32_t long_cap;
    // "all" mode (fused walk): t holds ONE table (the one-pass automaton of host/fused.hpp) that every line walks; no buckets,
    // no records — work item i = lines [i * kCapItemLines, ...) of line_off, ext_id / hist are written for every line
    uint32_t prefer_threads;     // CTA size the caller measured best for this work-item order (0 = by resident warps); GORP_TAIL_THREADS wins
    uint32_t all;
    uint32_t item_lines;         // lines per work item in "all" mode (<= kCapItemLines; smaller for small batches: enough items for every CTA)
    int64_t n_lines;
};
size_t tailwalk_smem_bytes(const TailDev&, int threads);
void k4c_tailwalk(const Launch&, const TailWalkParams&);

// result assembly of a batch that is pipelined in pieces: dst[i] = src[i] + bias ; dst[i] += src[i]
void k_bias_copy(const Launch&, int64_t* dst, const int64_t* src, int64_t n, int64_t bias);
void k_accumulate(const Launch&, int64_t* dst, const int64_t* src, int n);
// dst[i] = src[i] (ISO-8859-1 byte -> UTF-16 unit); both 16-byte aligned
void k_widen_latin1(const Launch&, const uint8_t* src, uint16_t* dst, int64_t n);

// UTF-8 ingest (kernels/utf8.cu): src = well-formed UTF-8 bytes (16-byte aligned), dst = the UTF-16 units they decode to.
// count: tile_counts[utf8_tiles(n)] = UTF-16 units per 4096-byte tile, *first_bad = offset of the first malformed byte (preset
// to ~0 by the caller); write: tile_base = exclusive scan of tile_counts.
int64_t utf8_tiles(int64_t n_bytes);
// slice_units (lines form, else nullptr): [ceil(n / 16)] units of the 4096-byte tile before each 16-byte slice
void k_utf8_count(const Launch&, const uint8_t* src, int64_t n, uint32_t* tile_counts, unsigned long long* first_bad, uint16_t* slice_units = nullptr);
void k_utf8_write(const Launch&, const uint8_t* src, int64_t n, const int64_t* tile_base, uint16_t* dst);
// Byte coordinates of the UTF-8 input (gorp_extract_text_utf8_bytes), kernels/utf8.cu.
// Count pass of K1 over the bytes (utf8_nl_count_mask_kernel): tile_counts[ceil(n / kNlTile)], masks[ceil(n / kNlTile) * 256]
// in the layout of k1_count_newlines_masks, so k1_scatter_masks(masks, n, ...) writes the byte line offsets (entries 1..).
void k_utf8_count_newlines_masks(const Launch&, const uint8_t* src, int64_t n, uint32_t* tile_counts, uint32_t* masks);
// Gather of one piece's rows in byte coordinates (utf8_rows_kernel): out_off[i] = byte start of line i + bias (i <= n_lines,
// out_off[n_lines] = end_off + bias), out_spans = the unit rows with every boundary moved to the byte offset of its sequence.
struct Utf8RowsParams {
    const uint8_t* bytes;        // the piece's UTF-8 bytes (16-byte aligned; read up to the 16-byte block of the last line's end)
    const int64_t* unit_off;     // [n_lines + 1] line offsets of the decoded piece (K1)
    const int64_t* byte_off;     // entries 1 .. of the byte line offsets (entry 0 is 0, entry n_lines is end_off)
    const int32_t* spans;        // [n_lines * stride] rows in unit offsets
    int64_t n_lines;
    int64_t end_off;             // n_bytes, + 1 when the piece does not end in '\n'
    int64_t bias;                // byte position of the piece in the caller's buffer
    uint32_t stride;             // <= 64
    int64_t* out_off;
    int32_t* out_spans;
};
// lines = true: the List<String> form over UTF-8 strings (gorp_extract_lines_utf8): no separator, byte_off is the caller's
// offsets [n_lines + 1] (the piece's bytes start at caller byte `bias`), out_off their copy (nullptr: not written); end_off
// is not used.
void k_utf8_rows(const Launch&, const Utf8RowsParams&, bool lines = false);
// Unit offsets of the strings of a UTF-8 piece (utf8_line_units_kernel): unit_off[i] = UTF-16 units of the decoded piece
// before byte byte_off[i] - base, from the count pass's tile_base (scanned) and slice_units; an interior offset that cuts a
// sequence or starts with a continuation byte sets first_bad (atomicMin) to the byte at which a string fails on its own.
// order_bad (or nullptr): set (atomicMin, preset to ~0) to the first i with byte_off[i + 1] < byte_off[i]; offsets outside
// [base, base + n] are not dereferenced.
void k_utf8_line_units(const Launch&, const uint8_t* src, int64_t n, const int64_t* byte_off, int64_t n_off, int64_t base, const int64_t* tile_base,
                       const uint16_t* slice_units, int64_t* unit_off, unsigned long long* first_bad, unsigned long long* order_bad = nullptr);

// matchAll (kernels/matchall.cu): the reference's own tables on the device
struct MatchAllDev {
    const uint16_t* classmap;    // [65536] Automata._alphabet
    const int32_t* trans;        // [S * C]  Automata._transitions, -1 = dead
    const uint32_t* accept_off;  // [S + 1]  CSR of Automata._accept
    const int32_t* accept_list;
    uint32_t n_classes;
};
void k_matchall_walk(const Launch&, const MatchAllDev&, const uint16_t* text, const int64_t* off, int64_t n_lines, int32_t* state, uint32_t* count);
void k_matchall_fill(const Launch&, const MatchAllDev&, const int32_t* state, const int64_t* out_off, int64_t n_lines, int32_t* out);

// Simulating Pike VM for extractions whose capture automaton could not be determinised (kernels/pike.cu)
struct PikeExtDev {
    uint32_t inst_off;    // of the extraction's n_insts + 1 entries in clo_off
    uint32_t n_insts, n_slots;
    uint32_t acc_off;     // of its n_insts * n_classes bytes in accepts
    uint32_t enabled;     // 0: the extraction has a real capture automaton
};
struct PikeDev {
    const PikeExtDev* ext;             // [E]
    const uint32_t* clo_off;           // closure CSR (global indexes into clo_target / clo_mask)
    const int32_t* clo_target;
    const unsigned long long* clo_mask;
    const uint8_t* accepts;
    const uint16_t* cls;               // [65536] unit -> symbol class of the capture side
    uint32_t n_classes, pair_hi_class;
    uint32_t max_insts, max_slots;
    uint32_t enabled;
};
size_t pike_scratch_ints_per_thread(const PikeDev&);
// decides the lines that came out as CAPTURE_FAIL(e) for an extraction e with P.ext[e].enabled: MATCH (ext_id, spans, histogram
// are patched) or a real capture failure (left as they are). scratch: scratch_threads * pike_scratch_ints_per_thread ints.
void k_pike_fixup(const Launch&, const PikeDev&, const uint16_t* text, const int64_t* line_off, int sep, int64_t n_lines, uint32_t span_stride,
                  int32_t* ext_id, int32_t* spans, unsigned long long* hist, uint32_t n_ext, int32_t* scratch, uint32_t scratch_threads);

// Value tables of a device-resident result (kernels/tables.cu, gorp_extract_tables_device). Positions of table e in the
// call's buffers, all in elements; entry E of the layout array holds the totals.
struct TableLayout {
    int64_t n_rows;              // matched lines of extraction e
    int64_t row_base;            // of its row indexes (multiple of 8)
    int64_t off_base;            // of column 0's offset segment; column k at off_base + k * seg
    int64_t seg;                 // offset entries per column: round_up(n_rows + 1, 8)
    int64_t valid_base;          // u32 words of column 0's bitmap; column k at valid_base + k * vwords
    int64_t vwords;              // round_up(ceil(n_rows / 32), 16)
    int64_t len_task, gather_task;  // first task of the table in the length and gather passes
    int64_t col_base;            // index of column 0 among all columns
    int64_t n_cols;              // groups of e
};
int64_t tables_tile_lines(uint32_t n_ext);  // lines per tile of the count / scatter passes
// counts[e * n_tiles + t] = lines of extraction e in tile t
void k_tables_count(const Launch&, const int32_t* ext_id, int64_t n_lines, uint32_t n_ext, int64_t tile_lines, int64_t n_tiles, uint32_t* counts);
// starts = exclusive scan of counts; slots[e] = 2 * groups of e (ignored when !with_groups: every table has 0 columns)
void k_tables_layout(const Launch&, const int64_t* starts, int64_t n_tiles, uint32_t n_ext, const uint32_t* slots, bool with_groups,
                     TableLayout* lay);
void k_tables_scatter(const Launch&, const int32_t* ext_id, int64_t n_lines, uint32_t n_ext, int64_t tile_lines, int64_t n_tiles,
                      const int64_t* starts, const TableLayout* lay, int64_t* rows);
// lens[lay.off_base total], valid (zeroed by the caller), stats[2 * columns] (zeroed: value units, nulls)
void k_tables_len(const Launch&, const TableLayout* lay, uint32_t n_ext, const int64_t* rows, const int32_t* spans, uint32_t stride,
                  uint32_t* lens, uint32_t* valid, unsigned long long* stats);
// offs = scan of lens; col_info[2 * col] = offs at the column's entry 0, col_info[2 * col + 1] = byte offset of its data
void k_tables_gather(const Launch&, const TableLayout* lay, uint32_t n_ext, const int64_t* rows, const int64_t* line_off, const int32_t* spans,
                     uint32_t stride, const void* text, int unit_bytes, const uint32_t* lens, int64_t* offs, const int64_t* col_info, uint8_t* data);
// The merge of one device's tables into the tables of a host call on several devices: n int64 entries of src plus `add`
// (row indexes, offsets; src may be dst), or with shift 1..7 a validity bitmap of n bits moved up by `shift` bits into
// (n + shift + 7) / 8 bytes of dst (the bits below `shift` of byte 0 are 0: the host ORs that byte into the bitmap).
struct RebaseJob {
    const void* src;
    void* dst;
    int64_t n;
    int64_t add;
    int64_t shift;
    int64_t first_block;  // blocks of the jobs before this one (tables_rebase_blocks)
};
int64_t tables_rebase_blocks(const RebaseJob&);
void k_tables_rebase(const Launch&, const RebaseJob* jobs, uint32_t n_jobs, int64_t n_blocks);

// K3: per-extraction histogram (E entries, then MISS, then capture failures).
void k3_histogram(const Launch&, const int32_t* ext_id, int64_t n_lines, uint32_t n_ext, unsigned long long* hist);

}  // namespace gorp
