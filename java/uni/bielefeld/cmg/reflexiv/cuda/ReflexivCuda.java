/*
 * ReflexivCuda -- Panama (java.lang.foreign, Java 22) binding of libreflexiv_cuda, include/reflexiv_cuda.h.
 *
 * NOT COMPILED IN THIS REPOSITORY'S BUILD IMAGE: it has no JDK (java, javac and jni.h are absent), so this file ships as
 * source only.  The same call sequences are built and tested from C++ (reflexiv_b200/csrc/reflexiv_main.cpp) and from
 * Python / ctypes (reflexiv_b200/_lib.py, pipeline.py); INTEGRATION.md explains where this class plugs into the
 * reference (pipeline/ReflexivDSMain.java:188-354, pipeline/ReflexivDataFrameCounter.java:178-233,
 * pipeline/ReflexivDSKmerLeftAndRightSorting.java:168-240).
 *
 * Ownership: every buffer handed to the library is caller owned and not retained; results are copied into buffers
 * allocated here.  One instance per driver thread.  Errors surface as RuntimeException carrying rfx_last_error().
 */
package uni.bielefeld.cmg.reflexiv.cuda;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemoryLayout;
import java.lang.foreign.MemoryLayout.PathElement;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.StructLayout;
import java.lang.foreign.SymbolLookup;
import java.lang.invoke.MethodHandle;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_BYTE;
import static java.lang.foreign.ValueLayout.JAVA_DOUBLE;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

import uni.bielefeld.cmg.reflexiv.util.DefaultParam;

public final class ReflexivCuda implements AutoCloseable {
    /** rfx_fastq_mode */
    public static final int FASTQ_RUN = 0, FASTQ_COUNTER = 1, FASTQ_LINE = 2;

    private static final Linker LINKER = Linker.nativeLinker();
    private static final SymbolLookup LIB = SymbolLookup.libraryLookup(System.getProperty("reflexiv.cuda.lib", "libreflexiv_cuda.so"), Arena.global());

    private static MethodHandle h(String name, FunctionDescriptor d) {
        return LINKER.downcallHandle(LIB.find(name).orElseThrow(() -> new UnsatisfiedLinkError(name)), d);
    }

    /** struct rfx_params (include/reflexiv_cuda.h): 18 x int32, 2 x int64 */
    static final StructLayout PARAMS = MemoryLayout.structLayout(
        JAVA_INT.withName("struct_size"), JAVA_INT.withName("kmer_size"), JAVA_INT.withName("min_kmer_coverage"),
        JAVA_INT.withName("max_kmer_coverage"), JAVA_INT.withName("min_error_coverage"), JAVA_INT.withName("min_contig"),
        JAVA_INT.withName("front_clip"), JAVA_INT.withName("end_clip"), JAVA_INT.withName("bubble"),
        JAVA_INT.withName("min_iter"), JAVA_INT.withName("max_iter"), JAVA_INT.withName("partitions"),
        JAVA_INT.withName("shuffle_partitions"), JAVA_INT.withName("counter_mode"), JAVA_INT.withName("fastq_mode"),
        JAVA_INT.withName("device"), JAVA_INT.withName("minimizer_len"), JAVA_INT.withName("reserved0"),
        JAVA_LONG.withName("table_capacity"), JAVA_LONG.withName("bin_target_kmers"));

    private static final MethodHandle PARAMS_DEFAULT = h("rfx_params_default", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle CREATE = h("rfx_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle DESTROY = h("rfx_destroy", FunctionDescriptor.ofVoid(ADDRESS));
    private static final MethodHandle LAST_ERROR = h("rfx_last_error", FunctionDescriptor.of(ADDRESS, ADDRESS));
    private static final MethodHandle PUSH_FASTQ = h("rfx_push_fastq", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG));
    private static final MethodHandle COUNT = h("rfx_count", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle COUNTS_SIZE = h("rfx_counts_size", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle COUNTS_COPY = h("rfx_counts_copy", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle COUNTS_CSV = h("rfx_counts_csv", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    private static final MethodHandle LOAD_COUNTS = h("rfx_load_counts", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG));
    private static final MethodHandle LOAD_COUNTS_CSV = h("rfx_load_counts_csv", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, JAVA_INT));
    private static final MethodHandle ASSEMBLE = h("rfx_assemble", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle CONTIGS_SIZE = h("rfx_contigs_size", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle CONTIGS_COPY = h("rfx_contigs_copy", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle STITCH_BEGIN = h("rfx_stitch_begin", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle STITCH_FINISH = h("rfx_stitch_finish", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle SORT_KMERS = h("rfx_sort_kmers", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_DOUBLE, JAVA_INT));
    private static final MethodHandle SORTED_CSV = h("rfx_sorted_csv", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    // multi-GPU over peer memory (include/reflexiv_cuda.h: rfx_shard_*): one ReflexivCuda per GPU, collective calls from one thread each
    private static final MethodHandle SHARD_INIT = h("rfx_shard_init", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_LONG));
    private static final MethodHandle SHARD_EXPORT = h("rfx_shard_export", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle SHARD_CONNECT = h("rfx_shard_connect", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT));
    private static final MethodHandle COUNT_SHARDED = h("rfx_count_sharded", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle SHARD_TABLE = h("rfx_shard_table", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle ASSEMBLE_SHARDED = h("rfx_assemble_sharded", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle SORT_KMERS_SHARDED = h("rfx_sort_kmers_sharded", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_DOUBLE, JAVA_INT));
    public static final int SHARD_HANDLE_BYTES = 128;

    /** One contig as the reference's DSKmerToContig sees it: bases plus the two end flags of the header. */
    public record Contig(String bases, int left, int right) {}

    private final Arena arena = Arena.ofConfined();
    private final MemorySegment ctx;
    private final int kmerSize;

    private static void setInt(MemorySegment prm, String field, int value) {
        prm.set(JAVA_INT, PARAMS.byteOffset(PathElement.groupElement(field)), value);
    }

    /** counterMode: `reflexiv counter` (coverage bounds applied as ReflexivDataFrameCounter.java:202-210 does), else `reflexiv run`. */
    public ReflexivCuda(DefaultParam p, boolean counterMode, int device) {
        this.kmerSize = p.kmerSize;
        try {
            MemorySegment prm = arena.allocate(PARAMS);
            check((int) PARAMS_DEFAULT.invoke(prm), MemorySegment.NULL);
            setInt(prm, "kmer_size", p.kmerSize);
            setInt(prm, "min_kmer_coverage", p.minKmerCoverage);
            setInt(prm, "max_kmer_coverage", p.maxKmerCoverage);
            setInt(prm, "min_error_coverage", p.minErrorCoverage);
            setInt(prm, "min_contig", p.minContig);
            setInt(prm, "front_clip", p.frontClip);
            setInt(prm, "end_clip", p.endClip);
            setInt(prm, "bubble", p.bubble ? 1 : 0);
            setInt(prm, "min_iter", p.minimumIteration);
            setInt(prm, "max_iter", p.maximumIteration);
            setInt(prm, "partitions", p.partitions);
            setInt(prm, "shuffle_partitions", p.shufflePartition);
            setInt(prm, "counter_mode", counterMode ? 1 : 0);
            setInt(prm, "fastq_mode", counterMode ? ("line".equals(p.inputFormat) ? FASTQ_LINE : FASTQ_COUNTER) : FASTQ_RUN);
            setInt(prm, "device", device);
            MemorySegment out = arena.allocate(ADDRESS);
            check((int) CREATE.invoke(out, prm), MemorySegment.NULL);
            ctx = out.get(ADDRESS, 0);
        } catch (RuntimeException | Error e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }

    /** Decompressed FASTQ text of one input file (a mapped file or a direct buffer); ends on a record boundary. */
    public void pushFastq(MemorySegment text) { call(() -> (int) PUSH_FASTQ.invoke(ctx, text, text.byteSize())); }

    /** extraction + groupBy.count + coverage filter (ReflexivDataFrameCounter.java:195-210, ReflexivDSMain.java:204-216) */
    public void count() { call(() -> (int) COUNT.invoke(ctx)); }

    /** fork filters + reflexible extension to the fixed point (ReflexivDSMain.java:221-338) */
    public void assemble() { call(() -> (int) ASSEMBLE.invoke(ctx)); }

    /**
     * -stitch (ReflexivDSMain.java:585-672): assembles with every record kept and builds the probe table of the thinly covered contig
     * ends; until {@link #stitchFinish()} every pushFastq scans reads for bridging fragments instead of storing them.
     */
    public void stitchBegin() { call(() -> (int) STITCH_BEGIN.invoke(ctx)); }

    /** Joins contig + fragment + contig chains; {@link #contigs()} then returns the stitched set. */
    public void stitchFinish() { call(() -> (int) STITCH_FINISH.invoke(ctx)); }

    /**
     * Ranks of one JVM: {@code ranks[r]} was created on device r.  Puts every rank's buffers into an arena, hands every rank the
     * handles of all ranks; afterwards {@link #countSharded()} / {@link #assembleSharded()} are collective calls, one thread per rank
     * (an ExecutorService with ranks.length threads), and {@link #countsCsv()} / {@link #contigs()} return what the rank owns.
     */
    public static void connect(ReflexivCuda[] ranks, long arenaBytes) {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment handles = a.allocate((long) ranks.length * SHARD_HANDLE_BYTES);
            for (int r = 0; r < ranks.length; r++) {
                final int rank = r;
                ranks[r].call(() -> (int) SHARD_INIT.invoke(ranks[rank].ctx, rank, ranks.length, arenaBytes));
                ranks[r].call(() -> (int) SHARD_EXPORT.invoke(ranks[rank].ctx, handles.asSlice((long) rank * SHARD_HANDLE_BYTES, SHARD_HANDLE_BYTES)));
            }
            for (ReflexivCuda k : ranks) k.call(() -> (int) SHARD_CONNECT.invoke(k.ctx, handles, ranks.length));
        }
    }

    /** collective: every rank calls it from its own thread */
    public void countSharded() { call(() -> (int) COUNT_SHARDED.invoke(ctx)); }

    /** collective, after every rank loaded any slice of a Count_k table (loadCounts, may be empty): afterwards this rank holds
     *  the rows whose minimiser bin it owns, as after countSharded(), and assembleSharded() follows */
    public void shardTable() { call(() -> (int) SHARD_TABLE.invoke(ctx)); }

    /** collective: every rank calls it from its own thread */
    public void assembleSharded() { call(() -> (int) ASSEMBLE_SHARDED.invoke(ctx)); }

    /** The rows of Count_<k>: `KMER,count\n`, formatted on the device. */
    public byte[] countsCsv() { return csv(COUNTS_CSV); }

    /** Keys in the reference's layout (k/32+1 longs for k > 31, else one), counts in countsOut[0]. */
    public long[][] counts(int[][] countsOut) {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment n = a.allocate(JAVA_LONG), w = a.allocate(JAVA_INT);
            check((int) COUNTS_SIZE.invoke(ctx, n, w), ctx);
            long rows = n.get(JAVA_LONG, 0);
            int words = w.get(JAVA_INT, 0);
            MemorySegment keys = a.allocate(JAVA_LONG, Math.max(1, rows * words)), cnt = a.allocate(JAVA_INT, Math.max(1, rows));
            check((int) COUNTS_COPY.invoke(ctx, keys, cnt), ctx);
            countsOut[0] = cnt.asSlice(0, rows * 4).toArray(JAVA_INT);
            long[] flat = keys.asSlice(0, rows * words * 8).toArray(JAVA_LONG);
            long[][] r = new long[(int) rows][words];
            for (int i = 0; i < rows; i++) System.arraycopy(flat, i * words, r[i], 0, words);
            return r;
        } catch (RuntimeException | Error e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }

    /** -kmerc: rows of an existing Count_<k> table, keys in the layout counts() returns (KmerBinarizer, ReflexivDSMain.java:3872-3948). */
    public void loadCounts(long[] keysFlat, int[] counts) {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment k = a.allocateFrom(JAVA_LONG, keysFlat), c = a.allocateFrom(JAVA_INT, counts);
            check((int) LOAD_COUNTS.invoke(ctx, k, c, (long) counts.length), ctx);
        } catch (RuntimeException | Error e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }

    /**
     * -kmerc: Count_<k> text (a mapped part file or a direct buffer, whole lines) parsed on the device; rows with
     * minCount <= count <= maxCount are kept in text order, behind the current table if append (include/reflexiv_cuda.h).
     */
    public void loadCountsCsv(MemorySegment text, long minCount, long maxCount, boolean append) {
        call(() -> (int) LOAD_COUNTS_CSV.invoke(ctx, text, text.byteSize(), minCount, maxCount, append ? 1 : 0));
    }

    /** Both strands of every contig, order unspecified (as the reference's part files). */
    public Contig[] contigs() {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment n = a.allocate(JAVA_LONG), tot = a.allocate(JAVA_LONG);
            check((int) CONTIGS_SIZE.invoke(ctx, n, tot), ctx);
            int nc = (int) n.get(JAVA_LONG, 0);
            long total = tot.get(JAVA_LONG, 0);
            MemorySegment bases = a.allocate(Math.max(1, total)), offs = a.allocate(JAVA_LONG, nc + 1L);
            MemorySegment left = a.allocate(JAVA_INT, Math.max(1, nc)), right = a.allocate(JAVA_INT, Math.max(1, nc));
            check((int) CONTIGS_COPY.invoke(ctx, bases, offs, left, right), ctx);
            Contig[] out = new Contig[nc];
            for (int i = 0; i < nc; i++) {
                long b = offs.getAtIndex(JAVA_LONG, i), e = offs.getAtIndex(JAVA_LONG, i + 1);
                String s = new String(bases.asSlice(b, e - b).toArray(JAVA_BYTE), java.nio.charset.StandardCharsets.US_ASCII);
                out[i] = new Contig(s, left.getAtIndex(JAVA_INT, i), right.getAtIndex(JAVA_INT, i));
            }
            return out;
        } catch (RuntimeException | Error e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }

    /** Count_<k>_sorted (ReflexivDSKmerLeftAndRightSorting.java:105-243): rows `KMER,1|left|right\n`. */
    public byte[] sortedCsv(int minErrorCoverage, double minRepeatFold, int maxKmerSize) {
        call(() -> (int) SORT_KMERS.invoke(ctx, minErrorCoverage, minRepeatFold, maxKmerSize));
        return csv(SORTED_CSV);
    }

    /** collective Count_<k>_sorted on a sharded table (after countSharded() or shardTable()): every rank calls it from its own
     *  thread and gets the rows of its own shard; their union is what sortedCsv() gives on one context holding the whole table */
    public byte[] sortKmersSharded(int minErrorCoverage, double minRepeatFold, int maxKmerSize) {
        call(() -> (int) SORT_KMERS_SHARDED.invoke(ctx, minErrorCoverage, minRepeatFold, maxKmerSize));
        return csv(SORTED_CSV);
    }

    public int kmerSize() { return kmerSize; }

    // ---- plumbing ----
    @FunctionalInterface private interface Call { int run() throws Throwable; }

    private void call(Call c) {
        try {
            check(c.run(), ctx);
        } catch (RuntimeException | Error e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }

    private byte[] csv(MethodHandle fn) {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment n = a.allocate(JAVA_LONG);
            check((int) fn.invoke(ctx, MemorySegment.NULL, 0L, n), ctx);
            long bytes = n.get(JAVA_LONG, 0);
            if (bytes == 0) return new byte[0];
            MemorySegment out = a.allocate(bytes);
            check((int) fn.invoke(ctx, out, bytes, n), ctx);
            return out.toArray(JAVA_BYTE);
        } catch (RuntimeException | Error e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }

    private static void check(int rc, MemorySegment c) throws Throwable {
        if (rc == 0) return;
        MemorySegment msg = (MemorySegment) LAST_ERROR.invoke(c);
        String text = msg.equals(MemorySegment.NULL) ? "" : msg.reinterpret(4096).getString(0);
        throw new RuntimeException("libreflexiv_cuda " + rc + ": " + text);
    }

    @Override public void close() {
        try {
            DESTROY.invoke(ctx);
        } catch (Throwable ignored) {
            // nothing to report on the way out
        }
        arena.close();
    }
}
