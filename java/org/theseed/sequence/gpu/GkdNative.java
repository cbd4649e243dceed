package org.theseed.sequence.gpu;

/**
 * JNI declarations for libgkd.so (include/gkd.h).  One native method per C entry point the
 * replacement processors need; handles are opaque longs, errors come back as negative status codes
 * (gkd_status) and are turned into exceptions by {@link GpuKmerEngine}.  Every method that fills a
 * Java array checks the array length against what the native call will write and returns GKD_EINVAL
 * (-1) on a mismatch.
 *
 * Not compiled in the build image (no JDK there; java/jni/gkd_jni.c is syntax-checked against a stub
 * jni.h by tests/test_abi_cpu.py); see INTEGRATION.md for the build line.
 */
final class GkdNative {
    static {
        System.loadLibrary("gkd_jni"); // links against libgkd.so
    }

    private GkdNative() { }

    static native long create(int device, int k, int alphabet, int strandMode);
    static native void destroy(long ctx);
    static native String lastError(long ctx);
    /** one genome / record from contigs (Latin-1 bytes); returns the set id or a negative status */
    static native int addSequences(long ctx, byte[][] contigs);
    /** every record of a FASTA file; returns {firstId, count} or null on error */
    static native int[] addFastaFile(long ctx, String path, boolean perRecord);
    static native String label(long ctx, int id);
    static native String comment(long ctx, int id);
    /** number of sets in the context */
    static native int count(long ctx);
    static native int buildSets(long ctx);
    static native int truncate(long ctx, int keep);
    /** fills dist (length count) with pairs [first, first+count) of the row-major strict upper triangle of n sets */
    static native int allVsAllRange(long ctx, int n, long first, long count, double[] dist);
    /** fills dist (length q.length * r.length, row-major) */
    static native int queryVsRef(long ctx, int[] q, int[] r, double[] dist);
    /** pairs [first, first+count) of the same enumeration whose distance is &lt;= maxDist, in order: the first
     *  min(total, cap) go to a, b (set ids, a &lt; b) and dist, cap being the shortest of the three arrays; returns the
     *  total number of such pairs (which may exceed cap) or a negative status */
    static native long allVsAllRangeWithin(long ctx, int n, long first, long count, double maxDist, int[] a, int[] b,
                                           double[] dist);
    /** every query's &lt;= k nearest references within maxDist, ascending distance, ties by position in r: refPos and
     *  dist (length q.length * k, row-major; unused slots -1 and -1.0), nFound (length q.length) */
    static native int queryVsRefNearest(long ctx, int[] q, int[] r, int k, double maxDist, boolean excludeSelf,
                                        int[] refPos, double[] dist, int[] nFound);
    /** each of the first n sets' &lt;= k nearest other sets within maxDist, ascending distance, ties by the smaller id;
     *  every pair is intersected once: pos and dist (length n * k, row-major; unused slots -1 and -1.0), nFound
     *  (length n) */
    static native int allVsAllNearest(long ctx, int n, int k, double maxDist, int[] pos, double[] dist, int[] nFound);
    /** single-linkage clusters of the first n sets at maxDist: label (length n) receives the smallest id of each set's
     *  cluster */
    static native int allVsAllClusters(long ctx, int n, double maxDist, int[] label);
    /** the single-linkage hierarchy of the first n sets up to maxDist: the minimum spanning forest of the pairs within
     *  maxDist in merge order; a, b, dist (length n - 1) receive its edges (a &lt; b), nEdges[0] their number */
    static native int allVsAllLinkage(long ctx, int n, double maxDist, int[] a, int[] b, double[] dist, int[] nEdges);
    /** the complete- (method 1) or average-linkage (method 2, UPGMA) hierarchy of the first n sets up to maxDist: a, b,
     *  height, size (length n - 1) receive the merges in order (a &lt; b the clusters' smallest ids, size the merged
     *  cluster's), nMerges[0] their number */
    static native int allVsAllAgglomerate(long ctx, int n, int method, double maxDist, int[] a, int[] b, double[] height,
                                          int[] size, int[] nMerges);
    static native int allVsAllCompleteLinkage(long ctx, int n, double maxDist, int[] a, int[] b, double[] height, int[] size,
                                              int[] nMerges);
    /** the neighbour-joining tree of the first n sets, rooted at the midpoint of its last edge: a, b, lenA, lenB (length
     *  n - 1) receive the joins in order (a &lt; b the joined subtrees' smallest ids, lenA and lenB their branch
     *  lengths), nJoins[0] their number */
    static native int allVsAllNj(long ctx, int n, int[] a, int[] b, double[] lenA, double[] lenB, int[] nJoins);
    /** the BIONJ tree of the first n sets, in the joins of allVsAllNj */
    static native int allVsAllBionj(long ctx, int n, int[] a, int[] b, double[] lenA, double[] lenB, int[] nJoins);
    /** the NJ (start 1) or BIONJ (start 2) tree of the first n sets refined by balanced minimum-evolution NNIs, in the
     *  joins of allVsAllNj; nSwaps[0] receives the number of swaps */
    static native int allVsAllBme(long ctx, int n, int start, int[] a, int[] b, double[] lenA, double[] lenB, int[] nJoins,
                                  long[] nSwaps);
    /** SequenceKmers.similarity / distance for one pair; either output may be null (length-1 arrays) */
    static native int pair(long ctx, int a, int b, long[] inter, double[] dist);
    /** out[0] = the reference's HashSet size of set id */
    static native int setSize(long ctx, int id, long[] out);
}
