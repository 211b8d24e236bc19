/*
 * Columnar view of one batch call of libgorpcuda (JDK 22+; NOT compiled or tested in this repository's build
 * environment: no JVM exists there — see INTEGRATION.md).
 *
 * Gorp.extract builds one ExtractionResult per line: an object, a String per group and (on asMap) a LinkedHashMap
 * (ExtractionResult.java:29-37, 65-88). For 10^8 lines that is 10^9 allocations and dwarfs the GPU time. A batch keeps the
 * result columns the native call returned — extraction index, line offsets, fixed-stride span rows — in heap arrays and
 * materialises an ExtractionResult only for the lines the caller asks for, through the same public
 * CookedExtraction.constructMatch(String, String[]) (model/CookedExtraction.java:54-57) the per-line path ends in.
 */
package com.salesforce.gorp.cuda;

import java.util.AbstractList;
import java.util.List;
import java.util.function.LongFunction;

import com.salesforce.gorp.ExtractionException;
import com.salesforce.gorp.ExtractionResult;
import com.salesforce.gorp.model.CookedExtraction;

public final class ExtractionBatch {
    /** extraction index per line: >= 0 matched, -1 miss (Gorp.extract returns null), <= -2: capture failure of extraction -2-e */
    public final int[] extId;
    /** UTF-16 unit offsets of the lines in the batch text ('\n'-separated forms: line i = [lineOff[i], lineOff[i+1] - 1)); byte
     *  offsets in the caller's buffer for a byte-coordinate batch ({@link GorpCuda#extractBatchUtf8Bytes}; for
     *  {@link GorpCuda#extractBatchUtf8Lines} line i = [lineOff[i], lineOff[i+1]), no separator), spans too */
    public final long[] lineOff;
    /** spanStride ints per line: (start, end) of group 1..n relative to the line start, -1 = group did not participate */
    public final int[] spans;
    public final int spanStride;
    /** per extraction, then misses, then capture failures */
    public final long[] histogram;

    private final CookedExtraction[] extractions;
    private final int[] groups;
    private final LongFunction<String> lines;
    private final ByteSource bytes;
    private final int sep;  // units between a line's end and the next line's start in a byte-coordinate batch ('\n': 1, strings: 0)

    /** Decodes bytes [from, to) of the caller's buffer (byte-coordinate batches). */
    interface ByteSource { String decode(long from, long to); }

    ExtractionBatch(int[] extId, long[] lineOff, int[] spans, int spanStride, long[] histogram, CookedExtraction[] extractions,
                    int[] groups, LongFunction<String> lines) {
        this(extId, lineOff, spans, spanStride, histogram, extractions, groups, lines, null);
    }

    ExtractionBatch(int[] extId, long[] lineOff, int[] spans, int spanStride, long[] histogram, CookedExtraction[] extractions,
                    int[] groups, LongFunction<String> lines, ByteSource bytes) {
        this(extId, lineOff, spans, spanStride, histogram, extractions, groups, lines, bytes, 1);
    }

    ExtractionBatch(int[] extId, long[] lineOff, int[] spans, int spanStride, long[] histogram, CookedExtraction[] extractions,
                    int[] groups, LongFunction<String> lines, ByteSource bytes, int sep) {
        this.extId = extId;
        this.lineOff = lineOff;
        this.spans = spans;
        this.spanStride = spanStride;
        this.histogram = histogram;
        this.extractions = extractions;
        this.groups = groups;
        this.lines = lines;
        this.bytes = bytes;
        this.sep = sep;
    }

    public int size() { return extId.length; }

    public boolean isMatch(int i) { return extId[i] >= 0; }

    public boolean isCaptureFailure(int i) { return extId[i] <= -2; }

    /** The matched extraction of line i, or null (miss / capture failure). */
    public CookedExtraction extraction(int i) { return extId[i] >= 0 ? extractions[extId[i]] : null; }

    /** Text of line i (decoded lazily from the caller's buffer). */
    public String line(int i) { return bytes != null ? bytes.decode(lineOff[i], lineOff[i + 1] - sep) : lines.apply(i); }

    /** Text [a, b) of line i: a substring of the line, or in a byte-coordinate batch the decoded bytes [start + a, start + b). */
    private String cut(int i, String line, int a, int b) {
        return bytes != null ? bytes.decode(lineOff[i] + a, lineOff[i] + b) : line.substring(a, b);
    }

    /** Value of capture group g (0-based) of line i without building an ExtractionResult; null when absent. */
    public String value(int i, int g) {
        if (extId[i] < 0 || g >= groups[extId[i]]) return null;
        int a = spans[i * spanStride + 2 * g], b = spans[i * spanStride + 2 * g + 1];
        return a < 0 ? null : cut(i, bytes != null ? null : line(i), a, b);
    }

    /** What Gorp.extract(line i) returns: null for a miss; throws for a capture failure (Gorp.java:173-177). */
    public ExtractionResult get(int i) throws ExtractionException { return get(i, false); }

    /** What Gorp.extractSafe(line i) returns: capture failures become null (Gorp.java:178-185). */
    public ExtractionResult getSafe(int i) {
        try {
            return get(i, true);
        } catch (ExtractionException e) {
            throw new IllegalStateException(e);  // cannot happen with safe == true
        }
    }

    private ExtractionResult get(int i, boolean safe) throws ExtractionException {
        final int e = extId[i];
        if (e == -1) return null;
        final String input = line(i);
        if (e < -1) {
            if (safe) return null;
            CookedExtraction x = extractions[-2 - e];
            throw new ExtractionException(input, String.format(
                    "Internal error: high-level match for extraction #%d (%s) failed to match generated regexp: %s",
                    -2 - e, x.getName(), x.getRegexpDesc()));
        }
        String[] values = new String[groups[e]];
        for (int g = 0; g < values.length; ++g) {
            int a = spans[i * spanStride + 2 * g], b = spans[i * spanStride + 2 * g + 1];
            values[g] = a < 0 ? null : cut(i, input, a, b);
        }
        return extractions[e].constructMatch(input, values);
    }

    /** Lazy List view with extractSafe semantics per element (nothing is materialised until get(i)). */
    public List<ExtractionResult> asList() {
        return new AbstractList<ExtractionResult>() {
            @Override public ExtractionResult get(int i) { return getSafe(i); }
            @Override public int size() { return extId.length; }
        };
    }
}
