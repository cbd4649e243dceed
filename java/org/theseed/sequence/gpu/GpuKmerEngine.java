package org.theseed.sequence.gpu;

import java.io.File;
import java.io.IOException;
import java.nio.charset.StandardCharsets;
import java.util.HashMap;
import java.util.List;
import java.util.Map;

import org.theseed.basic.ParseFailureException;

/**
 * Batched GPU replacement for the k-mer objects of org.theseed.sequence: the processors hand it whole
 * sequence lists and receive distance blocks, instead of calling SequenceKmers.distance() per pair.
 * The drop-in classes org.theseed.sequence.{KmerType,SequenceKmers,GenomeKmers,ProteinKmers} are handles
 * into the engine returned by {@link #shared(int, int)}.
 *
 * K is per engine (the reference keeps it in the statics GenomeKmers.setKmerSize /
 * ProteinKmers.setKmerSize, GenomeProcessor.java:86, ProteinKmerReader.java:92).
 */
public class GpuKmerEngine implements AutoCloseable {

    /** KmerType ordinal mapping used by the native side */
    public static final int DNA = 0, PROT = 1, RNA = 2;

    /** one engine per (alphabet, K) for the object-style API, so objects of one kind can be compared */
    private static final Map<Long, GpuKmerEngine> SHARED = new HashMap<Long, GpuKmerEngine>();

    private long ctx;
    /** sets added since the last build (built lazily by the first distance request) */
    private boolean dirty;

    public GpuKmerEngine(int alphabet, int kmerSize, int device) throws ParseFailureException {
        this.ctx = GkdNative.create(device, kmerSize, alphabet, 0);
        if (this.ctx == 0)
            throw new ParseFailureException(GkdNative.lastError(0));
        this.dirty = false;
    }

    /** @return the process-wide engine for this alphabet and kmer size (device 0) */
    public static synchronized GpuKmerEngine shared(int alphabet, int kmerSize) {
        long key = ((long) alphabet << 32) | (kmerSize & 0xFFFFFFFFL);
        GpuKmerEngine retVal = SHARED.get(key);
        if (retVal == null) {
            try {
                retVal = new GpuKmerEngine(alphabet, kmerSize, 0);
            } catch (ParseFailureException e) {
                throw new IllegalArgumentException(e.getMessage());
            }
            SHARED.put(key, retVal);
        }
        return retVal;
    }

    /** KmerType.createKmers(seq, K) / new ProteinKmers(str): returns the handle of the new set */
    public synchronized int add(String sequence) {
        this.dirty = true;
        return check(GkdNative.addSequences(this.ctx, new byte[][] { sequence.getBytes(StandardCharsets.ISO_8859_1) }));
    }

    /** new GenomeKmers(genome): one piece per contig; k-mers never span contigs */
    public synchronized int addGenome(List<String> contigs) {
        byte[][] parts = new byte[contigs.size()][];
        for (int i = 0; i < parts.length; i++)
            parts[i] = contigs.get(i).getBytes(StandardCharsets.ISO_8859_1);
        this.dirty = true;
        return check(GkdNative.addSequences(this.ctx, parts));
    }

    /** FastaInputStream(File): every record becomes a set; returns {firstId, count} */
    public synchronized int[] addFasta(File inFile) throws IOException {
        int[] r = GkdNative.addFastaFile(this.ctx, inFile.getPath(), true);
        if (r == null)
            throw new IOException(GkdNative.lastError(this.ctx));
        this.dirty = true;
        return r;
    }

    public String getLabel(int id) { return GkdNative.label(this.ctx, id); }
    public String getComment(int id) { return GkdNative.comment(this.ctx, id); }

    /** @return the number of sets in the engine */
    public int size() { return GkdNative.count(this.ctx); }

    /** build the sets of everything added since the last build (kernels 1-3) */
    public synchronized void build() {
        if (this.dirty) {
            check(GkdNative.buildSets(this.ctx));
            this.dirty = false;
        }
    }

    /** drop the sets with id &gt;= keep (e.g. query genomes that have been reported) */
    public synchronized void truncate(int keep) { check(GkdNative.truncate(this.ctx, keep)); }

    /** all pairs i &lt; j in list order, row-major strict upper triangle */
    public synchronized double[] allVsAll() {
        this.build();
        long n = this.size();
        long pairs = n * (n - 1) / 2;          // long arithmetic: n can exceed 65,536
        if (pairs > Integer.MAX_VALUE - 8)
            throw new IllegalArgumentException("Too many pairs for one array; use allVsAllRange in blocks.");
        double[] dist = new double[(int) pairs];
        check(GkdNative.allVsAllRange(this.ctx, (int) n, 0L, pairs, dist));
        return dist;
    }

    /** pairs [first, first + count) of the same enumeration, for reports larger than one Java array */
    public synchronized double[] allVsAllRange(long first, int count) {
        this.build();
        double[] dist = new double[count];
        check(GkdNative.allVsAllRange(this.ctx, this.size(), first, (long) count, dist));
        return dist;
    }

    /** every query against every reference, row-major */
    public synchronized double[] queryVsRef(int[] queries, int[] refs) {
        this.build();
        long cells = (long) queries.length * (long) refs.length;
        if (cells > Integer.MAX_VALUE - 8)
            throw new IllegalArgumentException("Too many pairs for one array; split the queries.");
        double[] dist = new double[(int) cells];
        check(GkdNative.queryVsRef(this.ctx, queries, refs, dist));
        return dist;
    }

    /** pairs i &lt; j of the first n sets within maxDist, in list order: {a, b} ids and their distances.  The triangle
     *  is read in ranges of at most rangePairs pairs; each range is selected on the GPU and only its hits come back. */
    public synchronized Within allVsAllWithin(double maxDist, int rangePairs) {
        this.build();
        long n = this.size();
        long pairs = n * (n - 1) / 2;
        Within out = new Within();
        int room = (int) Math.min(pairs, (long) rangePairs);
        int[] a = new int[room], b = new int[room];
        double[] dist = new double[room];
        for (long first = 0; first < pairs; first += rangePairs) {
            long count = Math.min((long) rangePairs, pairs - first);
            long hits = GkdNative.allVsAllRangeWithin(this.ctx, (int) n, first, count, maxDist, a, b, dist);
            if (hits < 0)
                check((int) hits);
            out.append(a, b, dist, (int) hits);  // hits <= count <= room: everything was written
        }
        return out;
    }

    /** the selected pairs of {@link #allVsAllWithin} */
    public static final class Within {
        public int[] a = new int[0], b = new int[0];
        public double[] dist = new double[0];
        public int size;

        void append(int[] xa, int[] xb, double[] xd, int n) {
            if (this.size + n > this.a.length) {
                int cap = Math.max(this.size + n, 2 * this.a.length);
                this.a = java.util.Arrays.copyOf(this.a, cap);
                this.b = java.util.Arrays.copyOf(this.b, cap);
                this.dist = java.util.Arrays.copyOf(this.dist, cap);
            }
            System.arraycopy(xa, 0, this.a, this.size, n);
            System.arraycopy(xb, 0, this.b, this.size, n);
            System.arraycopy(xd, 0, this.dist, this.size, n);
            this.size += n;
        }
    }

    /** every query's k nearest references within maxDist (ascending distance, ties by position in refs): refPos[i*k+j]
     *  is a position in refs, -1 in unused slots; returns the number found per query.  dist receives q.length * k values. */
    public synchronized int[] queryVsRefNearest(int[] queries, int[] refs, int k, double maxDist, boolean excludeSelf,
                                                int[] refPos, double[] dist) {
        this.build();
        int[] found = new int[queries.length];
        check(GkdNative.queryVsRefNearest(this.ctx, queries, refs, k, maxDist, excludeSelf, refPos, dist, found));
        return found;
    }

    /** the k-nearest-neighbour graph of every set (MashProcessor's getClosest, exact): pos[i*k+j] is the id of the
     *  j-th nearest other set of set i within maxDist (ascending distance, ties by the smaller id), -1 in unused slots;
     *  returns the number found per set.  pos and dist receive size() * k values. */
    public synchronized int[] allVsAllNearest(int k, double maxDist, int[] pos, double[] dist) {
        this.build();
        int n = this.size();
        int[] found = new int[n];
        check(GkdNative.allVsAllNearest(this.ctx, n, k, maxDist, pos, dist, found));
        return found;
    }

    /** single-linkage clusters of every set at maxDist (dereplication): two sets share a cluster when a chain of pairs,
     *  each with distance &lt;= maxDist, joins them; label[i] is the smallest id of set i's cluster, so label[i] == i
     *  marks a cluster's first member.  Every pair is intersected once and only the labels leave the GPU. */
    public synchronized int[] allVsAllClusters(double maxDist) {
        this.build();
        int[] label = new int[this.size()];
        check(GkdNative.allVsAllClusters(this.ctx, label.length, maxDist, label));
        return label;
    }

    /** the single-linkage hierarchy of every set up to maxDist (1.0: the whole tree): the merges of single-linkage
     *  agglomeration in order, i.e. the minimum spanning forest of the pairs within maxDist under (distance, a, b).
     *  a, b and dist (at least size() - 1 entries) receive the merged pair (a &lt; b) and its distance; returns the
     *  number of merges, size() minus the clusters at maxDist.  The clusters at any t &lt;= maxDist are the components
     *  of the merges with dist &lt;= t.  Every pair is intersected once and only the merges leave the GPU. */
    public synchronized int allVsAllLinkage(double maxDist, int[] a, int[] b, double[] dist) {
        this.build();
        int[] merges = new int[1];
        check(GkdNative.allVsAllLinkage(this.ctx, this.size(), maxDist, a, b, dist, merges));
        return merges[0];
    }

    /** linkage methods of allVsAllAgglomerate (gkd_link_method) */
    public static final int LINK_COMPLETE = 1, LINK_AVERAGE = 2;

    /** the complete- (LINK_COMPLETE) or average-linkage (LINK_AVERAGE, UPGMA) hierarchy of every set up to maxDist
     *  (1.0: the whole tree): the merges of the sequential agglomeration in order.  a, b, height and size (at least
     *  size() - 1 entries) receive the two clusters' smallest ids (a &lt; b), the cluster distance (average: rounded to
     *  the nearest double) and the merged cluster's size; returns the number of merges, size() minus the clusters at
     *  maxDist.  Every pair is intersected once; the distances stay on the GPU and only the merges leave it. */
    public synchronized int allVsAllAgglomerate(int method, double maxDist, int[] a, int[] b, double[] height, int[] size) {
        this.build();
        int[] merges = new int[1];
        check(GkdNative.allVsAllAgglomerate(this.ctx, this.size(), method, maxDist, a, b, height, size, merges));
        return merges[0];
    }

    /** allVsAllAgglomerate(LINK_COMPLETE, maxDist, ...), equal merge for merge, from the pairs within maxDist only: GPU
     *  memory grows with those pairs instead of with the square of size(), so it serves collections whose distance
     *  matrix does not fit on the GPU at dereplication thresholds. */
    public synchronized int allVsAllCompleteLinkage(double maxDist, int[] a, int[] b, double[] height, int[] size) {
        this.build();
        int[] merges = new int[1];
        check(GkdNative.allVsAllCompleteLinkage(this.ctx, this.size(), maxDist, a, b, height, size, merges));
        return merges[0];
    }

    /** the neighbour-joining tree of every set, rooted at the midpoint of its last edge: join t merges the current
     *  subtrees whose smallest ids are a[t] &lt; b[t], with branch lengths lenA[t] and lenB[t] from the new node (the
     *  arrays hold at least size() - 1 entries).  Returns the number of joins, size() - 1 (0 for fewer than two sets).
     *  Every pair is intersected once; the distances stay on the GPU and only the joins leave it. */
    public synchronized int allVsAllNj(int[] a, int[] b, double[] lenA, double[] lenB) {
        this.build();
        int[] joins = new int[1];
        check(GkdNative.allVsAllNj(this.ctx, this.size(), a, b, lenA, lenB, joins));
        return joins[0];
    }

    /** the BIONJ tree of every set, in the joins of allVsAllNj: BIONJ (Gascuel 1997) weights the two clusters of each
     *  join by a variance kept for every distance instead of NJ's one half each, which suits distances whose noise
     *  grows with the distance, such as Mash-style k-mer distances. */
    public synchronized int allVsAllBionj(int[] a, int[] b, double[] lenA, double[] lenB) {
        this.build();
        int[] joins = new int[1];
        check(GkdNative.allVsAllBionj(this.ctx, this.size(), a, b, lenA, lenB, joins));
        return joins[0];
    }

    /** the NJ (start 1) or BIONJ (start 2) tree of every set refined by balanced minimum-evolution nearest-neighbour
     *  interchanges (Desper and Gascuel 2002), with BME branch lengths, in the joins of allVsAllNj; returns the number of
     *  joins, and nSwaps[0] receives the number of swaps taken. */
    public synchronized int allVsAllBme(int start, int[] a, int[] b, double[] lenA, double[] lenB, long[] nSwaps) {
        this.build();
        int[] joins = new int[1];
        check(GkdNative.allVsAllBme(this.ctx, this.size(), start, a, b, lenA, lenB, joins, nSwaps));
        return joins[0];
    }

    /** SequenceKmers.distance(other) for the greedy callers (DistanceRepsProcessor, FastaDistanceRepsProcessor) */
    public synchronized double distance(int a, int b) {
        this.build();
        double[] out = new double[1];
        check(GkdNative.pair(this.ctx, a, b, null, out));
        return out[0];
    }

    /** SequenceKmers.similarity(other): kmers in common */
    public synchronized long similarity(int a, int b) {
        this.build();
        long[] inter = new long[1];
        check(GkdNative.pair(this.ctx, a, b, inter, null));
        return inter[0];
    }

    /** @return the reference's HashSet size of a set (both strands for DNA) */
    public synchronized long setSize(int id) {
        this.build();
        long[] out = new long[1];
        check(GkdNative.setSize(this.ctx, id, out));
        return out[0];
    }

    private int check(int rc) {
        if (rc < 0) {
            String msg = GkdNative.lastError(this.ctx);
            if (rc == -1) throw new IllegalArgumentException(msg);   // GKD_EINVAL
            throw new RuntimeException(msg);                          // GKD_ENOMEM / GKD_ECUDA / GKD_ESTATE
        }
        return rc;
    }

    @Override
    public synchronized void close() {
        if (this.ctx != 0) {
            GkdNative.destroy(this.ctx);
            this.ctx = 0;
        }
    }
}
