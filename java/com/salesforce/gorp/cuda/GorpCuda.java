/*
 * Panama FFM (java.lang.foreign, JDK 22+) binding of libgorpcuda.so — include/gorp_cuda.h.
 * NOT compiled or tested in this repository's build environment (no JVM there); see INTEGRATION.md.
 *
 * Batch counterpart of Gorp.extract(String) (Gorp.java:145-186): results are materialised through the public
 * CookedExtraction.constructMatch(String, String[]) (model/CookedExtraction.java:54-57), so ExtractionResult,
 * DefinitionReader and Gorp stay byte-for-byte what they are.
 */
package com.salesforce.gorp.cuda;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_CHAR;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemoryLayout;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.StructLayout;
import java.lang.foreign.SymbolLookup;
import java.lang.invoke.MethodHandle;
import java.nio.CharBuffer;
import java.util.ArrayList;
import java.util.List;

import com.salesforce.gorp.ExtractionException;
import com.salesforce.gorp.ExtractionResult;
import com.salesforce.gorp.Gorp;
import com.salesforce.gorp.model.CookedExtraction;

public final class GorpCuda implements AutoCloseable {
    private static final Linker LINKER = Linker.nativeLinker();
    private static final SymbolLookup LIB =
            SymbolLookup.libraryLookup(System.getProperty("gorp.cuda.lib", "libgorpcuda.so"), Arena.global());

    // struct gorp_result (include/gorp_cuda.h, ABI v2): { int64 n_lines; int32 n_extractions, span_stride; 4 pointers; void* owner; }
    private static final StructLayout RESULT = MemoryLayout.structLayout(
            JAVA_LONG.withName("n_lines"), JAVA_INT.withName("n_extractions"), JAVA_INT.withName("span_stride"),
            ADDRESS.withName("ext_id"), ADDRESS.withName("line_off"), ADDRESS.withName("spans"),
            ADDRESS.withName("histogram"), ADDRESS.withName("owner"));

    private static MethodHandle fn(String name, FunctionDescriptor d) {
        return LINKER.downcallHandle(LIB.find(name).orElseThrow(), d);
    }

    private static final MethodHandle ENGINE_CREATE = fn("gorp_engine_create",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, JAVA_INT, ADDRESS));
    private static final MethodHandle ENGINE_DESTROY = fn("gorp_engine_destroy", FunctionDescriptor.ofVoid(ADDRESS));
    private static final MethodHandle EXTRACT_LINES = fn("gorp_extract_lines",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    private static final MethodHandle EXTRACT_TEXT = fn("gorp_extract_text",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    private static final MethodHandle EXTRACT_TEXT_LATIN1 = fn("gorp_extract_text_latin1",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    private static final MethodHandle EXTRACT_TEXT_UTF8 = fn("gorp_extract_text_utf8",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    private static final MethodHandle EXTRACT_TEXT_UTF8_BYTES = fn("gorp_extract_text_utf8_bytes",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    private static final MethodHandle EXTRACT_LINES_UTF8 = fn("gorp_extract_lines_utf8",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    // struct gorp_match_result { int64 n_lines; const int64* accept_off; const int32* accept; void* owner; }
    private static final StructLayout MATCH_RESULT = MemoryLayout.structLayout(
            JAVA_LONG.withName("n_lines"), ADDRESS.withName("accept_off"), ADDRESS.withName("accept"), ADDRESS.withName("owner"));
    private static final MethodHandle MATCH_ALL_LINES = fn("gorp_match_all_lines",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    private static final MethodHandle MATCH_RESULT_RELEASE = fn("gorp_match_result_release", FunctionDescriptor.ofVoid(ADDRESS, ADDRESS));
    private static final MethodHandle RESULT_RELEASE = fn("gorp_result_release", FunctionDescriptor.ofVoid(ADDRESS, ADDRESS));
    private static final MethodHandle LAST_ERROR = fn("gorp_last_error", FunctionDescriptor.of(ADDRESS));

    private final Gorp gorp;
    private final CookedExtraction[] extractions;
    private final int[] groups;  // capture groups per extraction (JDKRegexpCookedExtraction._constructMatch reads groupCount())
    private final MemorySegment engine;

    public GorpCuda(Gorp gorp, int... devices) throws Throwable {
        this.gorp = gorp;
        this.extractions = gorp.getExtractions().toArray(new CookedExtraction[0]);
        this.groups = new int[extractions.length];
        for (int i = 0; i < groups.length; ++i)
            groups[i] = java.util.regex.Pattern.compile(extractions[i].getRegexpSource()).matcher("").groupCount();
        byte[] blob = DfaExport.export(gorp);
        try (Arena a = Arena.ofConfined()) {
            MemorySegment b = a.allocate(blob.length, 8);
            MemorySegment.copy(blob, 0, b, java.lang.foreign.ValueLayout.JAVA_BYTE, 0, blob.length);
            MemorySegment devs = devices.length == 0 ? MemorySegment.NULL : a.allocateFrom(JAVA_INT, devices);
            MemorySegment out = a.allocate(ADDRESS);
            check((int) ENGINE_CREATE.invokeExact(b, (long) blob.length, devs, devices.length, out));
            this.engine = out.get(ADDRESS, 0);
        }
    }

    /** Gorp.extractAll(List&lt;String&gt;): element null == miss; throws at the first capture failure (Gorp.java:173-177). */
    public List<ExtractionResult> extractAll(List<String> lines) throws Throwable {
        return extractAll(lines, false);
    }

    /** extractSafe semantics: capture failures become null (Gorp.java:178-185). */
    public List<ExtractionResult> extractAllSafe(List<String> lines) throws Throwable {
        return extractAll(lines, true);
    }

    private List<ExtractionResult> extractAll(List<String> lines, boolean safe) throws Throwable {
        final int n = lines.size();
        long units = 0;
        for (String s : lines) units += s.length();
        try (Arena a = Arena.ofConfined()) {
            MemorySegment text = a.allocate(Math.max(2 * units, 2), 16);
            MemorySegment off = a.allocate(8L * (n + 1), 8);
            long pos = 0;
            for (int i = 0; i < n; ++i) {
                String s = lines.get(i);
                off.setAtIndex(JAVA_LONG, i, pos);
                MemorySegment.copy(s.toCharArray(), 0, text, JAVA_CHAR, 2 * pos, s.length());
                pos += s.length();
            }
            off.setAtIndex(JAVA_LONG, n, pos);
            MemorySegment res = a.allocate(RESULT);
            check((int) EXTRACT_LINES.invokeExact(engine, text, off, (long) n, res));
            try {
                return materialise(res, i -> lines.get((int) i), n, safe);
            } finally {
                RESULT_RELEASE.invokeExact(engine, res);
            }
        }
    }

    /**
     * Gorp.extractAll(CharBuffer): '\n'-separated text. A direct buffer in NATIVE byte order is passed zero-copy; any
     * other buffer is copied char by char (ByteBuffer.allocateDirect(..).asCharBuffer() is BIG_ENDIAN by default: the
     * native side reads host-order UTF-16 and would see byte-swapped units).
     */
    public List<ExtractionResult> extractAll(CharBuffer text) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment seg;
            if (text.isDirect() && text.order() == java.nio.ByteOrder.nativeOrder()) {
                seg = MemorySegment.ofBuffer(text);
            } else {
                seg = a.allocate(Math.max(2L * text.remaining(), 2), 16);
                char[] tmp = new char[text.remaining()];
                text.duplicate().get(tmp);
                MemorySegment.copy(tmp, 0, seg, JAVA_CHAR, 0, tmp.length);
            }
            final CharBuffer view = text.duplicate();
            MemorySegment res = a.allocate(RESULT);
            check((int) EXTRACT_TEXT.invokeExact(engine, seg, (long) text.remaining(), res));
            try {
                long n = res.get(JAVA_LONG, 0);
                MemorySegment lineOff = res.get(ADDRESS, 24).reinterpret(8 * (n + 1));
                return materialise(res, i -> {
                    int s = (int) lineOff.getAtIndex(JAVA_LONG, i), e = (int) lineOff.getAtIndex(JAVA_LONG, i + 1) - 1;
                    return view.subSequence(s, e).toString();
                }, n, false);
            } finally {
                RESULT_RELEASE.invokeExact(engine, res);
            }
        }
    }

    /**
     * '\n'-separated log text held one byte per character (ISO-8859-1), e.g. a memory-mapped ASCII log file or
     * {@code String.getBytes(ISO_8859_1)} of LATIN1-coded Strings: half the bytes cross PCIe, results are those of
     * {@link #extractAll(CharBuffer)} on the same characters. A direct buffer is passed zero-copy.
     */
    public List<ExtractionResult> extractAllLatin1(java.nio.ByteBuffer text) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment seg;
            if (text.isDirect()) {
                seg = MemorySegment.ofBuffer(text);
            } else {
                seg = a.allocate(Math.max(text.remaining(), 1), 16);
                MemorySegment.copy(MemorySegment.ofBuffer(text), 0, seg, 0, text.remaining());
            }
            final java.nio.ByteBuffer view = text.duplicate();
            final int base = view.position();
            MemorySegment res = a.allocate(RESULT);
            check((int) EXTRACT_TEXT_LATIN1.invokeExact(engine, seg, (long) text.remaining(), res));
            try {
                long n = res.get(JAVA_LONG, 0);
                MemorySegment lineOff = res.get(ADDRESS, 24).reinterpret(8 * (n + 1));
                return materialise(res, i -> {
                    int s = (int) lineOff.getAtIndex(JAVA_LONG, i), e = (int) lineOff.getAtIndex(JAVA_LONG, i + 1) - 1;
                    byte[] b = new byte[e - s];
                    view.get(base + s, b);
                    return new String(b, java.nio.charset.StandardCharsets.ISO_8859_1);
                }, n, false);
            } finally {
                RESULT_RELEASE.invokeExact(engine, res);
            }
        }
    }

    /**
     * '\n'-separated log text as UTF-8 bytes (a log file as it is on disk, e.g. a memory-mapped file): decoded to UTF-16 on
     * the device; the columnar batch is what {@link #extractAll(CharBuffer)} would give on {@code new String(bytes, UTF_8)}.
     * Lines are decoded from the byte buffer only when asked for. Malformed UTF-8 fails the call.
     */
    public ExtractionBatch extractBatchUtf8(java.nio.ByteBuffer text) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment seg;
            if (text.isDirect()) {
                seg = MemorySegment.ofBuffer(text);
            } else {
                seg = a.allocate(Math.max(text.remaining(), 1), 16);
                MemorySegment.copy(MemorySegment.ofBuffer(text), 0, seg, 0, text.remaining());
            }
            final java.nio.ByteBuffer view = text.duplicate();
            MemorySegment res = a.allocate(RESULT);
            check((int) EXTRACT_TEXT_UTF8.invokeExact(engine, seg, (long) text.remaining(), res));
            try {
                // byte offsets of the lines (the native offsets count decoded UTF-16 units): one pass over the '\n' bytes
                final int n = (int) res.get(JAVA_LONG, 0);
                final int[] byteOff = new int[n + 1];
                int line = 0;
                final int base = view.position(), end = view.limit();
                for (int p = base; p < end && line < n; ++p) if (view.get(p) == 0x0A) byteOff[++line] = p + 1 - base;
                if (line < n) byteOff[n] = end - base + 1;  // last line not terminated
                return batch(res, n, i -> {
                    byte[] b = new byte[byteOff[(int) i + 1] - 1 - byteOff[(int) i]];
                    view.get(base + byteOff[(int) i], b);
                    return new String(b, java.nio.charset.StandardCharsets.UTF_8);
                });
            } finally {
                RESULT_RELEASE.invokeExact(engine, res);
            }
        }
    }

    /**
     * Same call as {@link #extractBatchUtf8}, with the results in BYTE coordinates of {@code text}: {@code lineOff} are byte
     * offsets relative to the buffer's position and spans byte offsets relative to the line start, so neither the lines nor
     * the offsets are rebuilt on the host; {@link ExtractionBatch#value} decodes only the value's bytes. Runs on all of the
     * engine's devices. Malformed UTF-8 fails the call.
     */
    public ExtractionBatch extractBatchUtf8Bytes(java.nio.ByteBuffer text) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment seg;
            if (text.isDirect()) {
                seg = MemorySegment.ofBuffer(text);
            } else {
                seg = a.allocate(Math.max(text.remaining(), 1), 16);
                MemorySegment.copy(MemorySegment.ofBuffer(text), 0, seg, 0, text.remaining());
            }
            final java.nio.ByteBuffer view = text.duplicate();
            final int base = view.position();
            MemorySegment res = a.allocate(RESULT);
            check((int) EXTRACT_TEXT_UTF8_BYTES.invokeExact(engine, seg, (long) text.remaining(), res));
            try {
                final int n = (int) res.get(JAVA_LONG, 0);
                return batch(res, n, null, (from, to) -> {
                    byte[] b = new byte[(int) (to - from)];
                    view.get(base + (int) from, b);
                    return new String(b, java.nio.charset.StandardCharsets.UTF_8);
                });
            } finally {
                RESULT_RELEASE.invokeExact(engine, res);
            }
        }
    }

    /**
     * Columnar batch over records held as UTF-8 bytes (a batch of Kafka records, a {@code List<byte[]>} of events): what
     * {@link #extractBatch(List)} gives on {@code new String(record, UTF_8)} for every record, in BYTE coordinates: lineOff
     * are offsets into the records laid end to end (record i = [lineOff[i], lineOff[i+1])), spans byte offsets relative to
     * the record's first byte. A '\n' inside a record is data. The records are copied to native memory as they are (no
     * decoding, no String per record) and decoded on the device; lines and values are decoded later from the records
     * themselves, which must not change while the batch is in use. Runs on all of the engine's devices. A record that is not
     * well-formed UTF-8 fails the call.
     */
    public ExtractionBatch extractBatchUtf8Lines(List<byte[]> records) throws Throwable {
        final int n = records.size();
        final long[] start = new long[n + 1];
        for (int i = 0; i < n; ++i) start[i + 1] = start[i] + records.get(i).length;
        try (Arena a = Arena.ofConfined()) {
            MemorySegment text = a.allocate(Math.max(start[n], 1), 16);
            MemorySegment off = a.allocate(8L * (n + 1), 8);
            for (int i = 0; i < n; ++i) {
                byte[] r = records.get(i);
                MemorySegment.copy(r, 0, text, java.lang.foreign.ValueLayout.JAVA_BYTE, start[i], r.length);
            }
            MemorySegment.copy(start, 0, off, JAVA_LONG, 0, n + 1);
            MemorySegment res = a.allocate(RESULT);
            check((int) EXTRACT_LINES_UTF8.invokeExact(engine, text, off, (long) n, res));
            try {
                // bytes [from, to) lie in one record: the first record that ends after `from` (the arena is gone by then)
                return batch(res, n, null, (from, to) -> {
                    if (to <= from) return "";
                    int lo = 0, hi = n;
                    while (lo < hi) {
                        int mid = (lo + hi) >>> 1;
                        if (start[mid + 1] <= from) lo = mid + 1;
                        else hi = mid;
                    }
                    return new String(records.get(lo), (int) (from - start[lo]), (int) (to - from), java.nio.charset.StandardCharsets.UTF_8);
                }, 0);
            } finally {
                RESULT_RELEASE.invokeExact(engine, res);
            }
        }
    }

    /** Columnar batch over a List&lt;String&gt; (Gorp.extractAll without materialising every ExtractionResult). */
    public ExtractionBatch extractBatch(List<String> lines) throws Throwable {
        final int n = lines.size();
        long units = 0;
        for (String s : lines) units += s.length();
        try (Arena a = Arena.ofConfined()) {
            MemorySegment text = a.allocate(Math.max(2 * units, 2), 16);
            MemorySegment off = a.allocate(8L * (n + 1), 8);
            long pos = 0;
            for (int i = 0; i < n; ++i) {
                String s = lines.get(i);
                off.setAtIndex(JAVA_LONG, i, pos);
                MemorySegment.copy(s.toCharArray(), 0, text, JAVA_CHAR, 2 * pos, s.length());
                pos += s.length();
            }
            off.setAtIndex(JAVA_LONG, n, pos);
            MemorySegment res = a.allocate(RESULT);
            check((int) EXTRACT_LINES.invokeExact(engine, text, off, (long) n, res));
            try {
                return batch(res, n, i -> lines.get((int) i));
            } finally {
                RESULT_RELEASE.invokeExact(engine, res);
            }
        }
    }

    /** PolyMatcher.match for a batch (Gorp.getMatcher().match(s) per string): all accepting indexes per string, ascending. */
    public int[][] matchAll(List<String> lines) throws Throwable {
        final int n = lines.size();
        long units = 0;
        for (String s : lines) units += s.length();
        try (Arena a = Arena.ofConfined()) {
            MemorySegment text = a.allocate(Math.max(2 * units, 2), 16);
            MemorySegment off = a.allocate(8L * (n + 1), 8);
            long pos = 0;
            for (int i = 0; i < n; ++i) {
                String s = lines.get(i);
                off.setAtIndex(JAVA_LONG, i, pos);
                MemorySegment.copy(s.toCharArray(), 0, text, JAVA_CHAR, 2 * pos, s.length());
                pos += s.length();
            }
            off.setAtIndex(JAVA_LONG, n, pos);
            MemorySegment res = a.allocate(MATCH_RESULT);
            check((int) MATCH_ALL_LINES.invokeExact(engine, text, off, (long) n, res));
            try {
                MemorySegment aoff = res.get(ADDRESS, 8).reinterpret(8L * (n + 1));
                long total = aoff.getAtIndex(JAVA_LONG, n);
                MemorySegment acc = res.get(ADDRESS, 16).reinterpret(4 * Math.max(total, 1));
                int[][] out = new int[n][];
                for (int i = 0; i < n; ++i) {
                    long a0 = aoff.getAtIndex(JAVA_LONG, i), a1 = aoff.getAtIndex(JAVA_LONG, i + 1);
                    out[i] = new int[(int) (a1 - a0)];
                    for (int k = 0; k < out[i].length; ++k) out[i][k] = acc.getAtIndex(JAVA_INT, a0 + k);
                }
                return out;
            } finally {
                MATCH_RESULT_RELEASE.invokeExact(engine, res);
            }
        }
    }

    /** Copies the native result columns into heap arrays (the native buffers go back to the engine's pool). */
    private ExtractionBatch batch(MemorySegment res, int n, java.util.function.LongFunction<String> lines) {
        return batch(res, n, lines, null);
    }

    /** With {@code bytes} (byte-coordinate results): lines and values are cut from the caller's buffer. */
    private ExtractionBatch batch(MemorySegment res, int n, java.util.function.LongFunction<String> lines, ExtractionBatch.ByteSource bytes) {
        return batch(res, n, lines, bytes, 1);
    }

    /** {@code sep}: bytes between a line's end and the next line's start ('\n'-separated text: 1, records: 0). */
    private ExtractionBatch batch(MemorySegment res, int n, java.util.function.LongFunction<String> lines, ExtractionBatch.ByteSource bytes, int sep) {
        final int stride = res.get(JAVA_INT, 12), nExt = res.get(JAVA_INT, 8);
        int[] extId = res.get(ADDRESS, 16).reinterpret(4L * Math.max(n, 1)).asSlice(0, 4L * n).toArray(JAVA_INT);
        long[] lineOff = res.get(ADDRESS, 24).reinterpret(8L * (n + 1)).toArray(JAVA_LONG);
        int[] spans = res.get(ADDRESS, 32).reinterpret(4L * Math.max((long) n * stride, 1)).asSlice(0, 4L * n * stride).toArray(JAVA_INT);
        long[] hist = res.get(ADDRESS, 40).reinterpret(8L * (nExt + 2)).toArray(JAVA_LONG);
        return new ExtractionBatch(extId, lineOff, spans, stride, hist, extractions, groups, lines, bytes, sep);
    }

    private interface LineSource { String line(long i); }

    private List<ExtractionResult> materialise(MemorySegment res, LineSource src, long n, boolean safe) throws ExtractionException {
        MemorySegment extId = res.get(ADDRESS, 16).reinterpret(4 * Math.max(n, 1));
        // one fixed row of span_stride int32 entries per line: (start, end) pairs of the matched extraction's groups
        long stride = res.get(JAVA_INT, 12);
        MemorySegment spans = res.get(ADDRESS, 32).reinterpret(4 * Math.max(n * stride, 1));
        List<ExtractionResult> out = new ArrayList<>((int) n);
        for (long i = 0; i < n; ++i) {
            int e = extId.getAtIndex(JAVA_INT, i);
            if (e == -1) { out.add(null); continue; }
            String input = src.line(i);
            if (e < -1) {
                if (safe) { out.add(null); continue; }
                CookedExtraction x = extractions[-2 - e];
                throw new ExtractionException(input, String.format(
                        "Internal error: high-level match for extraction #%d (%s) failed to match generated regexp: %s",
                        -2 - e, x.getName(), x.getRegexpDesc()));
            }
            long s0 = i * stride;
            String[] values = new String[groups[e]];
            for (int g = 0; g < values.length; ++g) {
                int a = spans.getAtIndex(JAVA_INT, s0 + 2L * g), b = spans.getAtIndex(JAVA_INT, s0 + 2L * g + 1);
                values[g] = a < 0 ? null : input.substring(a, b);
            }
            out.add(extractions[e].constructMatch(input, values));
        }
        return out;
    }

    private static void check(int rc) throws Throwable {
        if (rc == 0) return;
        MemorySegment msg = ((MemorySegment) LAST_ERROR.invokeExact()).reinterpret(4096);
        throw new IllegalStateException("libgorpcuda error " + rc + ": " + msg.getString(0));
    }

    @Override
    public void close() {
        try {
            ENGINE_DESTROY.invokeExact(engine);
        } catch (Throwable t) {
            throw new IllegalStateException(t);
        }
    }
}
