/* gkd_jni.c -- JNI glue between org.theseed.sequence.gpu.GkdNative and the C ABI of libgkd.so.
 * Build where a JDK exists (not in the build image; there it is syntax-checked against tests/stubs/jni.h):
 *   gcc -shared -fPIC -I$JAVA_HOME/include -I$JAVA_HOME/include/linux -Iinclude \
 *       java/jni/gkd_jni.c -Lgenome/distance_b200 -lgkd -o libgkd_jni.so
 * No callbacks into the JVM are made from CUDA threads.  Every Java array that a native call fills is
 * length-checked against what the call writes; status codes are returned, never swallowed. */
#include <jni.h>
#include <stdint.h>
#include <stdlib.h>

#include "gkd.h"

#define CTX(h) ((gkd_ctx *)(intptr_t)(h))
#define FN(name) Java_org_theseed_sequence_gpu_GkdNative_##name

JNIEXPORT jlong JNICALL FN(create)(JNIEnv *env, jclass c, jint device, jint k, jint alphabet, jint strand) {
    gkd_config cfg = {0};
    cfg.device = device;
    cfg.k = k;
    cfg.alphabet = alphabet;
    cfg.strand_mode = strand;
    gkd_ctx *ctx = NULL;
    (void)env;
    (void)c;
    return gkd_create(&ctx, &cfg) == GKD_OK ? (jlong)(intptr_t)ctx : 0;
}

JNIEXPORT void JNICALL FN(destroy)(JNIEnv *env, jclass c, jlong h) {
    (void)env;
    (void)c;
    gkd_destroy(CTX(h));
}

JNIEXPORT jstring JNICALL FN(lastError)(JNIEnv *env, jclass c, jlong h) {
    (void)c;
    return (*env)->NewStringUTF(env, gkd_last_error(CTX(h)));
}

JNIEXPORT jint JNICALL FN(addSequences)(JNIEnv *env, jclass c, jlong h, jobjectArray contigs) {
    (void)c;
    jsize n = (*env)->GetArrayLength(env, contigs);
    const char **ptrs = (const char **)calloc((size_t)n + 1, sizeof(char *));
    uint64_t *lens = (uint64_t *)calloc((size_t)n + 1, sizeof(uint64_t));
    jbyteArray *arrs = (jbyteArray *)calloc((size_t)n + 1, sizeof(jbyteArray));
    int rc = GKD_OK;
    uint32_t id = 0;
    jsize got = 0;
    if (!ptrs || !lens || !arrs) rc = GKD_ENOMEM;
    for (; rc == GKD_OK && got < n; got++) {
        arrs[got] = (jbyteArray)(*env)->GetObjectArrayElement(env, contigs, got);
        lens[got] = (uint64_t)(*env)->GetArrayLength(env, arrs[got]);
        ptrs[got] = (const char *)(*env)->GetByteArrayElements(env, arrs[got], NULL);
        if (!ptrs[got]) {
            rc = GKD_ENOMEM;
            break;
        }
    }
    /* the JVM's byte arrays are pageable memory: the library copies them before it returns */
    if (rc == GKD_OK) rc = gkd_add_sequences(CTX(h), ptrs, lens, (uint32_t)n, &id);
    for (jsize i = 0; i < got; i++) (*env)->ReleaseByteArrayElements(env, arrs[i], (jbyte *)ptrs[i], JNI_ABORT);
    free(ptrs);
    free(lens);
    free(arrs);
    return rc == GKD_OK ? (jint)id : rc;
}

JNIEXPORT jintArray JNICALL FN(addFastaFile)(JNIEnv *env, jclass c, jlong h, jstring path, jboolean perRecord) {
    (void)c;
    const char *p = (*env)->GetStringUTFChars(env, path, NULL);
    if (!p) return NULL;
    uint32_t first = 0, n = 0;
    int rc = gkd_add_fasta_file(CTX(h), p, perRecord ? 1 : 0, &first, &n);
    (*env)->ReleaseStringUTFChars(env, path, p);
    if (rc != GKD_OK) return NULL;
    jint out[2] = {(jint)first, (jint)n};
    jintArray r = (*env)->NewIntArray(env, 2);
    if (r) (*env)->SetIntArrayRegion(env, r, 0, 2, out);
    return r;
}

JNIEXPORT jstring JNICALL FN(label)(JNIEnv *env, jclass c, jlong h, jint id) {
    (void)c;
    return (*env)->NewStringUTF(env, gkd_label(CTX(h), (uint32_t)id));
}
JNIEXPORT jstring JNICALL FN(comment)(JNIEnv *env, jclass c, jlong h, jint id) {
    (void)c;
    return (*env)->NewStringUTF(env, gkd_comment(CTX(h), (uint32_t)id));
}

JNIEXPORT jint JNICALL FN(count)(JNIEnv *env, jclass c, jlong h) {
    (void)env;
    (void)c;
    return (jint)gkd_count(CTX(h));
}

JNIEXPORT jint JNICALL FN(buildSets)(JNIEnv *env, jclass c, jlong h) {
    (void)env;
    (void)c;
    return gkd_build_sets(CTX(h));
}

JNIEXPORT jint JNICALL FN(truncate)(JNIEnv *env, jclass c, jlong h, jint keep) {
    (void)env;
    (void)c;
    return keep < 0 ? GKD_EINVAL : gkd_truncate(CTX(h), (uint32_t)keep);
}

JNIEXPORT jint JNICALL FN(allVsAllRange)(JNIEnv *env, jclass c, jlong h, jint n, jlong first, jlong count,
                                         jdoubleArray dist) {
    (void)c;
    if (n < 0 || first < 0 || count < 0 || !dist) return GKD_EINVAL;
    /* the native call writes exactly `count` doubles: the Java array must hold them */
    if ((jlong)(*env)->GetArrayLength(env, dist) < count) return GKD_EINVAL;
    jdouble *d = (*env)->GetDoubleArrayElements(env, dist, NULL);
    if (!d) return GKD_ENOMEM;
    int rc = gkd_all_vs_all_range(CTX(h), (uint32_t)n, (uint64_t)first, (uint64_t)count, NULL, d);
    (*env)->ReleaseDoubleArrayElements(env, dist, d, 0);
    return rc;
}

JNIEXPORT jint JNICALL FN(queryVsRef)(JNIEnv *env, jclass c, jlong h, jintArray q, jintArray r, jdoubleArray dist) {
    (void)c;
    if (!q || !r || !dist) return GKD_EINVAL;
    jsize nq = (*env)->GetArrayLength(env, q), nr = (*env)->GetArrayLength(env, r);
    if ((jlong)(*env)->GetArrayLength(env, dist) < (jlong)nq * (jlong)nr) return GKD_EINVAL;
    jint *qa = (*env)->GetIntArrayElements(env, q, NULL);
    jint *ra = (*env)->GetIntArrayElements(env, r, NULL);
    jdouble *d = (*env)->GetDoubleArrayElements(env, dist, NULL);
    int rc = (qa && ra && d) ? gkd_query_vs_ref(CTX(h), (const uint32_t *)qa, (uint32_t)nq, (const uint32_t *)ra,
                                                (uint32_t)nr, NULL, d)
                             : GKD_ENOMEM;
    if (d) (*env)->ReleaseDoubleArrayElements(env, dist, d, 0);
    if (ra) (*env)->ReleaseIntArrayElements(env, r, ra, JNI_ABORT);
    if (qa) (*env)->ReleaseIntArrayElements(env, q, qa, JNI_ABORT);
    return rc;
}

JNIEXPORT jint JNICALL FN(pair)(JNIEnv *env, jclass c, jlong h, jint a, jint b, jlongArray inter, jdoubleArray dist) {
    (void)c;
    if (a < 0 || b < 0) return GKD_EINVAL;
    if ((inter && (*env)->GetArrayLength(env, inter) < 1) || (dist && (*env)->GetArrayLength(env, dist) < 1))
        return GKD_EINVAL;
    uint64_t I = 0;
    double d = 1.0;
    int rc = gkd_pair(CTX(h), (uint32_t)a, (uint32_t)b, &I, NULL, &d);
    if (rc != GKD_OK) return rc; /* a failed call is an error, never "distance 1.0" */
    if (inter) {
        jlong v = (jlong)I;
        (*env)->SetLongArrayRegion(env, inter, 0, 1, &v);
    }
    if (dist) (*env)->SetDoubleArrayRegion(env, dist, 0, 1, &d);
    return GKD_OK;
}

JNIEXPORT jint JNICALL FN(setSize)(JNIEnv *env, jclass c, jlong h, jint id, jlongArray out) {
    (void)c;
    if (id < 0 || !out || (*env)->GetArrayLength(env, out) < 1) return GKD_EINVAL;
    uint64_t n = 0;
    int rc = gkd_set_size(CTX(h), (uint32_t)id, &n, NULL, NULL);
    if (rc != GKD_OK) return rc;
    jlong v = (jlong)n;
    (*env)->SetLongArrayRegion(env, out, 0, 1, &v);
    return GKD_OK;
}

/* fills a/b/dist (each at least `cap` long, cap = the shortest of the three) with the first hits of the pairs
 * [first, first+count) within maxDist; returns the total number of hits (may exceed cap) or a negative status */
JNIEXPORT jlong JNICALL FN(allVsAllRangeWithin)(JNIEnv *env, jclass c, jlong h, jint n, jlong first, jlong count, jdouble maxDist,
                                               jintArray a, jintArray b, jdoubleArray dist) {
    (void)c;
    if (n < 0 || first < 0 || count < 0 || !a || !b || !dist) return GKD_EINVAL;
    jlong cap = (*env)->GetArrayLength(env, a);
    if ((jlong)(*env)->GetArrayLength(env, b) < cap) cap = (*env)->GetArrayLength(env, b);
    if ((jlong)(*env)->GetArrayLength(env, dist) < cap) cap = (*env)->GetArrayLength(env, dist);
    uint32_t *ha = (uint32_t *)malloc((size_t)cap * 4 + 4), *hb = (uint32_t *)malloc((size_t)cap * 4 + 4);
    double *hd = (double *)malloc((size_t)cap * 8 + 8);
    int rc = (ha && hb && hd) ? GKD_OK : GKD_ENOMEM;
    gkd_hits hits = {ha, hb, NULL, hd, (uint64_t)cap, 0};
    if (rc == GKD_OK) rc = gkd_all_vs_all_range_within(CTX(h), (uint32_t)n, (uint64_t)first, (uint64_t)count, maxDist, &hits);
    if (rc == GKD_OK) {
        /* the native call wrote min(n, cap) entries: exactly what the Java arrays receive */
        const jsize w = (jsize)((jlong)hits.n < cap ? (jlong)hits.n : cap);
        (*env)->SetIntArrayRegion(env, a, 0, w, (const jint *)ha);
        (*env)->SetIntArrayRegion(env, b, 0, w, (const jint *)hb);
        (*env)->SetDoubleArrayRegion(env, dist, 0, w, hd);
    }
    free(ha);
    free(hb);
    free(hd);
    return rc == GKD_OK ? (jlong)hits.n : (jlong)rc;
}

/* every query's k nearest references within maxDist: refPos / dist hold q.length * k entries, nFound q.length */
JNIEXPORT jint JNICALL FN(queryVsRefNearest)(JNIEnv *env, jclass c, jlong h, jintArray q, jintArray r, jint k, jdouble maxDist,
                                             jboolean excludeSelf, jintArray refPos, jdoubleArray dist, jintArray nFound) {
    (void)c;
    if (!q || !r || !refPos || !dist || !nFound || k < 1) return GKD_EINVAL;
    jsize nq = (*env)->GetArrayLength(env, q), nr = (*env)->GetArrayLength(env, r);
    const jlong slots = (jlong)nq * (jlong)k;
    if ((jlong)(*env)->GetArrayLength(env, refPos) < slots || (jlong)(*env)->GetArrayLength(env, dist) < slots ||
        (*env)->GetArrayLength(env, nFound) < nq)
        return GKD_EINVAL;
    jint *qa = (*env)->GetIntArrayElements(env, q, NULL);
    jint *ra = (*env)->GetIntArrayElements(env, r, NULL);
    jint *pos = (*env)->GetIntArrayElements(env, refPos, NULL);
    jint *found = (*env)->GetIntArrayElements(env, nFound, NULL);
    jdouble *d = (*env)->GetDoubleArrayElements(env, dist, NULL);
    int rc = (qa && ra && pos && found && d)
                 ? gkd_query_vs_ref_nearest(CTX(h), (const uint32_t *)qa, (uint32_t)nq, (const uint32_t *)ra, (uint32_t)nr,
                                            (uint32_t)k, maxDist, excludeSelf ? 1 : 0, (uint32_t *)pos, NULL, d,
                                            (uint32_t *)found)
                 : GKD_ENOMEM;
    if (d) (*env)->ReleaseDoubleArrayElements(env, dist, d, 0);
    if (found) (*env)->ReleaseIntArrayElements(env, nFound, found, 0);
    if (pos) (*env)->ReleaseIntArrayElements(env, refPos, pos, 0);
    if (ra) (*env)->ReleaseIntArrayElements(env, r, ra, JNI_ABORT);
    if (qa) (*env)->ReleaseIntArrayElements(env, q, qa, JNI_ABORT);
    return rc;
}

/* each of the first n sets' k nearest other sets within maxDist: pos / dist hold n * k entries, nFound n */
JNIEXPORT jint JNICALL FN(allVsAllNearest)(JNIEnv *env, jclass c, jlong h, jint n, jint k, jdouble maxDist, jintArray pos,
                                           jdoubleArray dist, jintArray nFound) {
    (void)c;
    if (!pos || !dist || !nFound || n < 0 || k < 1) return GKD_EINVAL;
    const jlong slots = (jlong)n * (jlong)k;
    if ((jlong)(*env)->GetArrayLength(env, pos) < slots || (jlong)(*env)->GetArrayLength(env, dist) < slots ||
        (*env)->GetArrayLength(env, nFound) < n)
        return GKD_EINVAL;
    jint *p = (*env)->GetIntArrayElements(env, pos, NULL);
    jint *found = (*env)->GetIntArrayElements(env, nFound, NULL);
    jdouble *d = (*env)->GetDoubleArrayElements(env, dist, NULL);
    gkd_neighbors out = {(uint32_t *)p, NULL, d, (uint32_t *)found};
    int rc = (p && found && d) ? gkd_all_vs_all_nearest(CTX(h), (uint32_t)n, (uint32_t)k, maxDist, &out) : GKD_ENOMEM;
    if (d) (*env)->ReleaseDoubleArrayElements(env, dist, d, 0);
    if (found) (*env)->ReleaseIntArrayElements(env, nFound, found, 0);
    if (p) (*env)->ReleaseIntArrayElements(env, pos, p, 0);
    return rc;
}

/* single-linkage clusters of the first n sets at maxDist: label holds n entries, the smallest id of each set's cluster */
JNIEXPORT jint JNICALL FN(allVsAllClusters)(JNIEnv *env, jclass c, jlong h, jint n, jdouble maxDist, jintArray label) {
    (void)c;
    if (!label || n < 0 || (*env)->GetArrayLength(env, label) < n) return GKD_EINVAL;
    jint *l = (*env)->GetIntArrayElements(env, label, NULL);
    int rc = l ? gkd_all_vs_all_clusters(CTX(h), (uint32_t)n, maxDist, (uint32_t *)l, NULL) : GKD_ENOMEM;
    if (l) (*env)->ReleaseIntArrayElements(env, label, l, 0);
    return rc;
}

/* the single-linkage hierarchy of the first n sets up to maxDist: a, b, dist hold n - 1 entries (the forest edges in
 * merge order); nEdges[0] receives their number */
JNIEXPORT jint JNICALL FN(allVsAllLinkage)(JNIEnv *env, jclass c, jlong h, jint n, jdouble maxDist, jintArray a,
                                           jintArray b, jdoubleArray dist, jintArray nEdges) {
    (void)c;
    if (!a || !b || !dist || !nEdges || n < 0 || (*env)->GetArrayLength(env, nEdges) < 1) return GKD_EINVAL;
    const jint cap = n > 0 ? n - 1 : 0;
    if ((*env)->GetArrayLength(env, a) < cap || (*env)->GetArrayLength(env, b) < cap ||
        (*env)->GetArrayLength(env, dist) < cap)
        return GKD_EINVAL;
    jint *pa = (*env)->GetIntArrayElements(env, a, NULL);
    jint *pb = (*env)->GetIntArrayElements(env, b, NULL);
    jdouble *d = (*env)->GetDoubleArrayElements(env, dist, NULL);
    gkd_hits out = {(uint32_t *)pa, (uint32_t *)pb, NULL, d, (uint64_t)cap, 0};
    int rc = (pa && pb && d) ? gkd_all_vs_all_linkage(CTX(h), (uint32_t)n, maxDist, &out) : GKD_ENOMEM;
    if (d) (*env)->ReleaseDoubleArrayElements(env, dist, d, 0);
    if (pb) (*env)->ReleaseIntArrayElements(env, b, pb, 0);
    if (pa) (*env)->ReleaseIntArrayElements(env, a, pa, 0);
    if (rc == GKD_OK) {
        jint ne = (jint)out.n;
        (*env)->SetIntArrayRegion(env, nEdges, 0, 1, &ne);
    }
    return rc;
}

/* the complete- (method 1) or average-linkage (method 2) hierarchy of the first n sets up to maxDist: a, b, height, size
 * hold n - 1 entries (the merges in order); nMerges[0] receives their number */
JNIEXPORT jint JNICALL FN(allVsAllAgglomerate)(JNIEnv *env, jclass c, jlong h, jint n, jint method, jdouble maxDist,
                                               jintArray a, jintArray b, jdoubleArray height, jintArray size,
                                               jintArray nMerges) {
    (void)c;
    if (!a || !b || !height || !size || !nMerges || n < 0 || (*env)->GetArrayLength(env, nMerges) < 1) return GKD_EINVAL;
    const jint cap = n > 0 ? n - 1 : 0;
    if ((*env)->GetArrayLength(env, a) < cap || (*env)->GetArrayLength(env, b) < cap ||
        (*env)->GetArrayLength(env, height) < cap || (*env)->GetArrayLength(env, size) < cap)
        return GKD_EINVAL;
    jint *pa = (*env)->GetIntArrayElements(env, a, NULL);
    jint *pb = (*env)->GetIntArrayElements(env, b, NULL);
    jdouble *ph = (*env)->GetDoubleArrayElements(env, height, NULL);
    jint *ps = (*env)->GetIntArrayElements(env, size, NULL);
    gkd_merges out = {(uint32_t *)pa, (uint32_t *)pb, ph, (uint32_t *)ps, (uint64_t)cap, 0};
    int rc = (pa && pb && ph && ps) ? gkd_all_vs_all_agglomerate(CTX(h), (uint32_t)n, method, maxDist, &out) : GKD_ENOMEM;
    if (ps) (*env)->ReleaseIntArrayElements(env, size, ps, 0);
    if (ph) (*env)->ReleaseDoubleArrayElements(env, height, ph, 0);
    if (pb) (*env)->ReleaseIntArrayElements(env, b, pb, 0);
    if (pa) (*env)->ReleaseIntArrayElements(env, a, pa, 0);
    if (rc == GKD_OK) {
        jint nm = (jint)out.n;
        (*env)->SetIntArrayRegion(env, nMerges, 0, 1, &nm);
    }
    return rc;
}
