/* libgorpcuda — C ABI of the B200 batch extraction engine for gorp definitions.
 *
 * Drop-in boundary (SURVEY.md §8b). Each entry point names the reference interface it replaces; paths are relative
 * to gorp-core/src/main/java/com/salesforce/gorp/ of salesforce/gorp.
 *
 *   reference (per line, JVM)                                  this library (per batch, GPU)
 *   --------------------------------------------------------   ------------------------------------------------
 *   DefinitionReader.reader(..).read()   DefinitionReader.java:51-84
 *   Gorp.construct(defs, cooker)         Gorp.java:50-92        gorp_compile_definition   (JVM-less hosts)
 *   Automata fields + regexp sources     autom/Automata.java:23-26,
 *                                        model/CookedExtraction.java:46   -> DfaExport blob -> gorp_engine_create
 *   PolyMatcher.match(CharSequence)      autom/PolyMatcher.java:123-133  \
 *   Gorp.extract(String)                 Gorp.java:145-186                > gorp_extract_lines / gorp_extract_text
 *   CookedExtraction.match(String)       jdkre/JDKRegexpCookedExtraction.java:36-59 /
 *   new ExtractionResult(...)            model/CookedExtraction.java:54-57   (Java materialises from gorp_result)
 *
 * Conventions: plain pointers and sizes, no exceptions cross the boundary; 0 = OK, < 0 = gorp_status; the message of
 * the last failure on the calling thread is gorp_last_error(). Text is UTF-16 code units in host byte order (Java
 * `char`). There is NO CPU fallback: every gorp_extract_* call fails with GORP_E_CUDA when no usable device exists.
 */
#ifndef GORP_CUDA_H
#define GORP_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GORP_ABI_VERSION 2

typedef enum gorp_status {
    GORP_OK = 0,
    GORP_E_ARG = -1,         /* null / out-of-range argument */
    GORP_E_DEFINITION = -2,  /* DefinitionParseException of the reference (DefinitionParseException.java:17) */
    GORP_E_UNSUPPORTED = -3, /* definition is legal for the reference but outside the GPU subset (DESIGN.md) */
    GORP_E_BLOB = -4,        /* malformed / corrupt DfaExport blob */
    GORP_E_CUDA = -5,        /* CUDA error or no device */
    GORP_E_OOM = -6,
    GORP_E_INTERNAL = -7
} gorp_status;

/* Per-line outcome codes in gorp_result.ext_id (Gorp.java:159-177):
 *   >= 0        index of the matched extraction (declaration order), spans present
 *   GORP_MISS   extract() would return null
 *   <= -2       extract() would throw ExtractionException for extraction index (-2 - ext_id):
 *               the combined DFA accepted but the java.util.regex dialect of that extraction did not */
#define GORP_MISS (-1)
#define GORP_CAPTURE_FAIL(e) (-2 - (e))

typedef struct gorp_engine gorp_engine;

typedef struct gorp_result {
    int64_t n_lines;
    int32_t n_extractions;
    int32_t span_stride;      /* int32 entries per result row of `spans` = 2 * (groups of the widest extraction) */
    const int32_t* ext_id;    /* [n_lines] */
    const int64_t* line_off;  /* [n_lines+1] start of each line in the caller's text; line i spans
                                 [line_off[i], line_off[i+1] - sep) with sep = 1 for gorp_extract_text ('\n'
                                 separated; line_off[n_lines] = n_units (+1 when the text does not end in '\n'))
                                 and sep = 0 for gorp_extract_lines (a copy of the caller's offsets) */
    const int32_t* spans;     /* [n_lines * span_stride] one fixed-size row per line: row i starts at i * span_stride
                                 and holds 2 * n_groups(ext_id[i]) valid entries = (start, end) pairs in UTF-16 units
                                 relative to the start of the line, in group order == extractor-name order; (-1,-1)
                                 when a group did not participate; the rest of the row, and the whole row of a MISS
                                 or capture-failed line, is -1. Fixed rows (instead of a CSR) keep the device path
                                 free of a span-offset prefix sum and let Java index rows directly. */
    const int64_t* histogram; /* [n_extractions + 2]: lines per extraction, then MISS, then capture failures */
    void* owner;              /* internal */
} gorp_result;

typedef struct gorp_blob_info {
    uint32_t n_states, n_classes, n_extractions, reserved;
} gorp_blob_info;

typedef struct gorp_extraction_info {  /* pointers stay valid as long as the blob they came from */
    uint32_t n_groups;
    uint32_t n_extractor_names;
    const uint16_t* name;            uint32_t name_len;
    const uint16_t* automaton_regex; uint32_t automaton_regex_len;  /* brics dialect, Gorp.java:68 */
    const uint16_t* jdk_regex;       uint32_t jdk_regex_len;        /* CookedExtraction.getRegexpSource() */
    const char* append_json;         uint32_t append_json_len;      /* raw `append` objects, '\n' separated */
} gorp_extraction_info;

int gorp_abi_version(void);
const char* gorp_last_error(void);
int gorp_device_count(void);

/* --- definition -> blob (host only; what DefinitionReader.read() + Gorp.construct() + DfaExport do in Java) */
int gorp_compile_definition(const char* grp_utf8, size_t len, void** blob, size_t* blob_len);
/* PolyMatcher.create(String...) for raw automaton-dialect patterns (autom/PolyMatcher.java:64-84): a blob whose
 * extractions have no capture groups (the JDK dialect string is left empty => match-only engine). */
int gorp_compile_patterns(const uint16_t* const* patterns, const uint32_t* lens, uint32_t n, void** blob, size_t* blob_len);
void gorp_blob_free(void* blob);

/* --- blob introspection (host only) */
int gorp_blob_get_info(const void* blob, size_t len, gorp_blob_info* out);
int gorp_blob_get_extraction(const void* blob, size_t len, uint32_t index, gorp_extraction_info* out);
int gorp_blob_get_extractor_name(const void* blob, size_t len, uint32_t extraction, uint32_t k,
                                 const uint16_t** name, uint32_t* name_len);
/* Raw tables exactly as Automata holds them (autom/Automata.java:23-26); accept lists as CSR. */
int gorp_blob_get_tables(const void* blob, size_t len, const uint16_t** classmap, const int32_t** transitions,
                         const int32_t** accept_first, const uint32_t** accept_off, const int32_t** accept_list);

/* --- engine: immutable after creation; concurrent gorp_extract_* calls on one engine are allowed */
int gorp_engine_create(const void* blob, size_t len, const int* devices, int n_devices, gorp_engine** out);
void gorp_engine_destroy(gorp_engine* e);

/* Gorp.extractAll(List<String>): `text` is the concatenation of the strings, off[i]..off[i+1] delimit string i. */
int gorp_extract_lines(gorp_engine* e, const uint16_t* text, const int64_t* off, int64_t n_lines, gorp_result* out);
/* Gorp.extractAll(CharBuffer): split on U+000A only; a final line without '\n' counts; '\r' is data. */
int gorp_extract_text(gorp_engine* e, const uint16_t* text, int64_t n_units, gorp_result* out);
/* Same call for text held as ISO-8859-1 bytes, one byte per character — what a JDK 9+ String with the LATIN1 coder holds
 * (java.lang.String compact strings; `String.getBytes(ISO_8859_1)` is a plain copy for such strings), i.e. the usual
 * case for log text. The bytes are widened to UTF-16 on the device, so the host-to-device copy moves half the bytes of
 * gorp_extract_text; results are identical to gorp_extract_text on the zero-extended text (spans and line_off count
 * characters == UTF-16 units). Split on byte 0x0A. */
int gorp_extract_text_latin1(gorp_engine* e, const uint8_t* text, int64_t n_bytes, gorp_result* out);
/* Same call for text held as UTF-8 bytes — log files as they are on disk (the reference reads UTF-8 the same way for its
 * definitions, io/InputLineReader.java:51; a Java caller would otherwise decode the bytes to Strings first). The bytes are
 * decoded to UTF-16 on the device (supplementary characters become surrogate pairs), so ASCII text crosses PCIe at one byte
 * per character. Results are those of gorp_extract_text on `new String(bytes, UTF_8)`: line_off and spans count UTF-16
 * units of the DECODED text. Split on byte 0x0A. The input must be well-formed UTF-8 (Unicode table 3-7): a malformed
 * sequence fails the call with GORP_E_ARG and the byte offset in gorp_last_error() — no replacement characters are
 * invented. Runs on the engine's first device. */
int gorp_extract_text_utf8(gorp_engine* e, const uint8_t* text, int64_t n_bytes, gorp_result* out);
/* Same call as gorp_extract_text_utf8, with the results in BYTE coordinates of the caller's buffer: line i is bytes
 * [line_off[i], line_off[i+1] - 1) (line_off[n_lines] = n_bytes, + 1 when the text does not end in '\n'), spans are
 * (start, end) byte offsets relative to the line's first byte. ext_id and histogram are those of gorp_extract_text_utf8.
 * Runs on all of the engine's devices (contiguous line-aligned byte ranges, rows concatenated in device order). */
int gorp_extract_text_utf8_bytes(gorp_engine* e, const uint8_t* text, int64_t n_bytes, gorp_result* out);
/* Gorp.extractAll(List<String>) for strings held as UTF-8 bytes, e.g. an Arrow/Parquet string column (int64 offsets) or a
 * batch of byte[] records: string i is bytes [off[i], off[i+1]) of `text`; a '\n' inside a string is data. Results are
 * those of gorp_extract_lines on the UTF-16 of `new String(bytes_i, UTF_8)` for every string, in BYTE coordinates:
 * line_off is a copy of `off` (sep = 0), spans are (start, end) byte offsets relative to the string's first byte;
 * ext_id and histogram are unchanged. Every string must be well-formed UTF-8 on its own (Unicode table 3-7): otherwise
 * GORP_E_ARG, "malformed UTF-8 at byte N", N = the lowest byte of `text` at which decoding some string on its own fails.
 * Bytes outside [off[0], off[n_lines]) are never read. Runs on all of the engine's devices. */
int gorp_extract_lines_utf8(gorp_engine* e, const uint8_t* text, const int64_t* off, int64_t n_lines, gorp_result* out);
void gorp_result_release(gorp_engine* e, gorp_result* r);

/* PolyMatcher.match for a batch (reference autom/PolyMatcher.java:123-133, reached through Gorp.getMatcher(), Gorp.java:135-137):
 * for every string ALL regex / extraction indexes whose automaton accepts the whole string, ascending (Automata.accept,
 * autom/Automata.java:137-139) — not only the first one the extract path uses. CSR: the indexes of string i are
 * accept[accept_off[i] .. accept_off[i+1]). Works on any engine (definitions and gorp_compile_patterns blobs). */
typedef struct gorp_match_result {
    int64_t n_lines;
    const int64_t* accept_off; /* [n_lines + 1] */
    const int32_t* accept;     /* [accept_off[n_lines]] */
    void* owner;
} gorp_match_result;
int gorp_match_all_lines(gorp_engine* e, const uint16_t* text, const int64_t* off, int64_t n_lines, gorp_match_result* out);
void gorp_match_result_release(gorp_engine* e, gorp_match_result* r);

/* --- device-resident variants: `d_text` (and `d_off`) already live in the HBM of the engine's device `dev_index`
 * (index into the `devices` array given at creation) and must be 16-byte aligned; only a 32-byte aligned `d_text` gets
 * the walkers that read 32-byte blocks (256-bit loads), any other takes the 16-byte-load kernels. Results stay in device memory
 * owned by the engine until the next call on the same (engine, dev_index). `stream` is a cudaStream_t (NULL = the
 * CUDA default stream, as everywhere in CUDA). The call enqueues the kernels on that stream; the text form waits once for the newline
 * count (it sizes the per-line arrays). Used by bench.py for the HBM-resident `value`. */
#define GORP_FLAG_SYNC 1          /* cudaStreamSynchronize before returning */
#define GORP_FLAG_TIME_KERNELS 2  /* bracket every kernel with CUDA events on `stream` (see gorp_kernel_times) */

typedef struct gorp_device_result {
    int64_t n_lines;
    int32_t span_stride;
    int32_t reserved;
    const int32_t* d_ext_id;
    const int64_t* d_line_off;
    const int32_t* d_spans;
    const int64_t* d_histogram;
    const int64_t* d_n_lines; /* device scalar */
} gorp_device_result;

int gorp_extract_text_device(gorp_engine* e, int dev_index, const uint16_t* d_text, int64_t n_units, void* stream,
                             int flags, gorp_device_result* out);
int gorp_extract_lines_device(gorp_engine* e, int dev_index, const uint16_t* d_text, const int64_t* d_off,
                              int64_t n_lines, void* stream, int flags, gorp_device_result* out);

/* The same device-resident calls for UTF-8 held in HBM: a log file read into device memory, a torch uint8 tensor, or a
 * cuDF / Arrow string column (its bytes plus int64 offsets; widen int32 offsets first). Results are in BYTE coordinates,
 * exactly those of gorp_extract_text_utf8_bytes (text form) and gorp_extract_lines_utf8 (lines form, d_line_off = the
 * caller's d_off) on the same bytes; ext_id and histogram are unchanged. Malformed UTF-8 fails with GORP_E_ARG and
 * "malformed UTF-8 at byte N" as in the host forms; in the lines form so do offsets that start below 0 or decrease
 * ("offsets must be non-decreasing (line i)", checked on the device), and bytes outside [d_off[0], d_off[n_lines]) are
 * never read. Conventions of the calls above (alignment, results, stream, flags). Host round trips: two per call —
 * text form: {decoded total, first malformed byte} and the newline count; lines form: {d_off[0], d_off[n_lines]} and
 * {decoded total, first malformed byte, first decreasing offset}. Engine scratch: the decoded UTF-16 text, 2 bytes per
 * input byte (n_bytes, or d_off[n_lines] - d_off[0]); the lines form also copies its bytes into the engine (1 byte per
 * byte), so that a first string at any byte offset meets the aligned kernels. */
int gorp_extract_text_utf8_device(gorp_engine* e, int dev_index, const uint8_t* d_text, int64_t n_bytes, void* stream, int flags,
                                  gorp_device_result* out);
int gorp_extract_lines_utf8_device(gorp_engine* e, int dev_index, const uint8_t* d_text, const int64_t* d_off, int64_t n_lines,
                                   void* stream, int flags, gorp_device_result* out);

/* What ExtractionResult.asMap() gives per line, as columns in device memory: one table per extraction, one string column per
 * extractor name, in Arrow layout (large_utf8 for the UTF-8 calls: 64-bit offsets, LSB-first validity bitmap), so that
 * Arrow's C data interface, cuDF or torch can wrap the buffers without copying.
 *
 * Source: the result of the last successful device-resident extract call on (e, dev_index) — gorp_extract_text_device,
 * gorp_extract_lines_device, gorp_extract_text_utf8_device or gorp_extract_lines_utf8_device. Every other extract or match
 * call that reaches the context (the host forms reuse the same result scratch, gorp_match_all_lines, a device-resident call
 * that fails) makes that result unreadable: the call then fails with GORP_E_ARG, as it does when no such call ran. A call
 * refused for its arguments before it reaches the context, gorp_kernel_times and this call itself leave the result readable.
 * The caller's d_text (and d_off of the lines forms) must hold the same contents, in stream order, until this call's kernels
 * have run: the values are read from there.
 *
 * Rows: table e holds exactly the lines with ext_id == e, in ascending line order (n_rows == histogram[e]); MISS and
 * CAPTURE_FAIL lines are in no table. Values: row r of column k, with span (s, t) of group k of the line, is code units
 * [line_off[line] + s, line_off[line] + t) of the caller's d_text, not transcoded — UTF-16 units (Java `char` data) after
 * the UTF-16 calls, bytes after the UTF-8 calls (every group boundary is a sequence start there, so each column is valid
 * UTF-8); offsets count the same units. A group that did not participate, (-1, -1), is a null: bit r of the bitmap is 0
 * and the value is empty. Bitmap padding bits are 0. An extraction without groups has 0 columns (null column arrays) and
 * only d_row; a table without rows has offsets {0} in every column.
 *
 * Every device buffer is 64-byte aligned. The tables stay valid until the next extract call on (e, dev_index); a second
 * tables call replaces them; the extract result they came from is not changed. Conventions of the device-resident calls
 * (stream, GORP_FLAG_SYNC, GORP_FLAG_TIME_KERNELS: stages tables_rank, tables_len, tables_scan, tables_gather). Host round
 * trips: one (the per-column totals that size the value buffers). Engine scratch: 8 B per line of the result (row
 * indexes) and 12 B per (line, group of the widest extraction) for lengths and the offset scan, then 8 B per value
 * (offsets), the values themselves and the bitmaps; plus 12 B per (extraction, tile of max(2048, 32 * extractions) lines). */
typedef struct gorp_value_table {       /* the lines of extraction e, in line order */
    int64_t n_rows;                     /* == histogram[e] of the call */
    int32_t n_columns;                  /* == groups of e; column k = extractor name k (gorp_blob_get_extractor_name(e, k)) */
    int32_t reserved;
    const int64_t* d_row;               /* [n_rows] index of the line in the call's result, strictly ascending */
    const int64_t* const* d_offsets;    /* host array [n_columns] of device pointers, each [n_rows + 1], offsets[0] = 0 */
    const void* const* d_data;          /* host array [n_columns] of device pointers: the values, concatenated */
    const uint8_t* const* d_valid;      /* host array [n_columns] of device pointers: Arrow validity bitmaps */
    const int64_t* null_count;          /* host [n_columns] */
} gorp_value_table;

/* (after gorp_extract_text_utf8_tables / gorp_extract_lines_utf8_tables every pointer here, d_row, d_offsets[k], d_data[k]
 * and d_valid[k] included, is a pinned HOST pointer) */
typedef struct gorp_device_tables {
    int32_t n_tables;                   /* == n_extractions; table e = extraction e */
    int32_t unit_bytes;                 /* 2 after the UTF-16 calls, 1 after the UTF-8 calls */
    const gorp_value_table* tables;     /* host array [n_tables] */
} gorp_device_tables;

int gorp_extract_tables_device(gorp_engine* e, int dev_index, void* stream, int flags, gorp_device_tables* out);

/* gorp_extract_text_utf8_bytes / gorp_extract_lines_utf8 that also return the values as tables in HOST memory — for callers
 * whose text is on the host (a log file, a batch of records, an Arrow or Parquet string column read on the CPU) and that
 * hand the values on as columns (Parquet, pandas, Arrow Java) rather than one string per group per line.
 *
 * *out is exactly what the plain call returns on the same arguments, and the call fails exactly where the plain call fails,
 * with the same status and message; a null `tables` is GORP_E_ARG. *tables follows the contract of
 * gorp_extract_tables_device with these differences: every pointer in it is pinned host memory; unit_bytes is 1; d_row
 * indexes rows of *out; the values are bytes [line_off[row] + s, line_off[row] + t) of the caller's `text`. Every buffer is
 * 64-byte aligned, bitmap padding bits are 0, an extraction without groups (and every extraction of a match-only engine,
 * gorp_compile_patterns) has rows and no columns. On several devices every table is still one table: device d's rows
 * follow those of the devices before it.
 *
 * The tables belong to the result: they stay valid until gorp_result_release(e, out), whatever other calls run on the
 * engine in between, and their pinned buffers return to the engine with the result (allocated on the NUMA node of the
 * engine's first device, as the rows are). Like every host call, these calls make the last device-resident result
 * unreadable for gorp_extract_tables_device.
 *
 * Cost on top of the plain call, per device: the device keeps its whole byte range of the batch in engine scratch (1 byte
 * per input byte; one device-to-device copy per staged piece), builds the tables of its rows after its last piece with the
 * stages and the engine scratch of gorp_extract_tables_device, and copies them to the host. Host round trips: one per
 * device (the per-column totals), then on several devices one synchronisation of all of them before the merge. Pinned
 * host memory: 8 B per matched line (row indexes), 8 B per (matched line, group) (offsets), the values, and the bitmaps,
 * each segment rounded up to 64 B. */
int gorp_extract_text_utf8_tables(gorp_engine* e, const uint8_t* text, int64_t n_bytes, gorp_result* out,
                                  gorp_device_tables* tables);
int gorp_extract_lines_utf8_tables(gorp_engine* e, const uint8_t* text, const int64_t* off, int64_t n_lines, gorp_result* out,
                                   gorp_device_tables* tables);

/* Device time per pipeline stage, summed over the calls made with GORP_FLAG_TIME_KERNELS on (e, dev_index) since the
 * last reset: names[i] / total_ms[i] for i < *n (at most `cap`), `calls` = timed calls, `launches` = kernels launched
 * by this context (all calls). Waits for the last timed call to finish. */
int gorp_kernel_times(gorp_engine* e, int dev_index, const char** names, double* total_ms, int cap, int* n,
                      int64_t* calls, int64_t* launches, int reset);

#ifdef __cplusplus
}
#endif
#endif /* GORP_CUDA_H */
