/*
 * ldagpu_jni.c -- JNI binding of libldagpu.so for JDK 8-21 (the reference builds with Java 8, pom.xml:152-154).
 *
 * java/cc/mallet/topics/GpuLDASampler.java in this repository calls the C ABI through the Panama FFM API
 * (JDK 22+).  On an older JDK the same class declares the calls as `private static native` methods of a
 * nested class `cc.mallet.topics.GpuLDASampler$Native` and loads this stub; the C signatures it forwards to
 * are exactly those of include/ldagpu.h.  NOT compiled in this repository's build image (no JDK, no jni.h).
 *
 *   gcc -shared -fPIC -I$JAVA_HOME/include -I$JAVA_HOME/include/linux -I../../include \
 *       ldagpu_jni.c -L<dir of libldagpu.so> -lldagpu -o libldagpu_jni.so
 *
 * Java side (excerpt):
 *   static final class Native {
 *       static { System.loadLibrary("ldagpu_jni"); }
 *       static native long   create(int K, int V, long D, long[] docOffsets, int[] tokens, double[] alpha,
 *                                   double beta, long seed, int scheme, int device, long docBase, long tokenBase);
 *       static native long   createMulti(int K, int V, long D, long[] docOffsets, int[] tokens, double[] alpha,
 *                                        double beta, long seed, int scheme, int[] devices);   // gpu_devices: one JVM, several GPUs
 *       static native void   setPhiSampler(long h, int sampler, int aliasPoissonThreshold);     // gpu_polyaurn
 *       static native void   destroy(long h);
 *       static native void   initZJavaRandom(long h, int seed);
 *       static native int    sweepGetZ(long h, int n, int[] z);          // returns the sweeps run
 *       static native void   setZ(long h, int[] z, boolean redrawPhi);
 *       static native void   getTypeTopicCounts(long h, int[] out);      // int[V*K], row-major [V][K]
 *       static native void   getTopicTotals(long h, int[] out);
 *       static native void   getPhi(long h, double[] out);               // double[K*V], row-major [K][V]
 *       static native double logLikelihood(long h);
 *       static native double logPosterior(long h);
 *       static native void   abort(long h);
 *       static native void   getCountHistograms(long h, long[] docTopicHist, long[] typeTopicHist);   // either may be empty
 *       static native void   setAlpha(long h, double[] alpha);           // optimizeAlpha / optimizeBeta (MSL:812-905)
 *       static native void   setBeta(long h, double beta);
 *       static native void   setTestDocuments(long h, long[] docOffsets, int[] tokens);   // addTestInstances
 *       static native double heldOutLogLikelihood(long h, int nParticles);            // evaluateLeftToRight
 *   }
 * Every failure is rethrown as IllegalStateException with ldagpu_last_error's message, which is what the
 * reference's own samplers throw on an invariant break (UncollapsedParallelLDA.java:475-481,1828-1830).
 */
#include <jni.h>
#include <stddef.h>
#include <stdint.h>

#include "ldagpu.h"

#define CLS(name) Java_cc_mallet_topics_GpuLDASampler_00024Native_##name

static void throw_last(JNIEnv *env, ldagpu_handle h)
{
    jclass ex = (*env)->FindClass(env, "java/lang/IllegalStateException");
    if (ex) (*env)->ThrowNew(env, ex, ldagpu_last_error(h));
}

JNIEXPORT jlong JNICALL CLS(create)(JNIEnv *env, jclass c, jint K, jint V, jlong D, jlongArray docOffsets,
                                    jintArray tokens, jdoubleArray alpha, jdouble beta, jlong seed, jint scheme,
                                    jint device, jlong docBase, jlong tokenBase)
{
    (void)c;
    ldagpu_handle h = NULL;
    jlong *off = (*env)->GetLongArrayElements(env, docOffsets, NULL);
    jint *tok = (*env)->GetIntArrayElements(env, tokens, NULL);
    jdouble *al = (*env)->GetDoubleArrayElements(env, alpha, NULL);
    int rc = ldagpu_create(K, V, D, (const int64_t *)off, (const int32_t *)tok, al, beta, (uint64_t)seed, scheme,
                           device, docBase, tokenBase, &h);
    (*env)->ReleaseLongArrayElements(env, docOffsets, off, JNI_ABORT);   /* the library has copied everything */
    (*env)->ReleaseIntArrayElements(env, tokens, tok, JNI_ABORT);
    (*env)->ReleaseDoubleArrayElements(env, alpha, al, JNI_ABORT);
    if (rc) { throw_last(env, NULL); return 0; }
    return (jlong)(intptr_t)h;
}

/* one JVM thread, several GPUs (the reference's coordinator thread, tui/ParallelLDA.java:173-202): the library shards the
 * corpus over `devices` and exchanges counts / Phi between them over NVLink peer memory */
JNIEXPORT jlong JNICALL CLS(createMulti)(JNIEnv *env, jclass c, jint K, jint V, jlong D, jlongArray docOffsets,
                                         jintArray tokens, jdoubleArray alpha, jdouble beta, jlong seed, jint scheme,
                                         jintArray devices)
{
    (void)c;
    ldagpu_handle h = NULL;
    jlong *off = (*env)->GetLongArrayElements(env, docOffsets, NULL);
    jint *tok = (*env)->GetIntArrayElements(env, tokens, NULL);
    jdouble *al = (*env)->GetDoubleArrayElements(env, alpha, NULL);
    jint *dev = (*env)->GetIntArrayElements(env, devices, NULL);
    int rc = ldagpu_create_multi(K, V, D, (const int64_t *)off, (const int32_t *)tok, al, beta, (uint64_t)seed, scheme,
                                 (*env)->GetArrayLength(env, devices), (const int32_t *)dev, &h);
    (*env)->ReleaseLongArrayElements(env, docOffsets, off, JNI_ABORT);
    (*env)->ReleaseIntArrayElements(env, tokens, tok, JNI_ABORT);
    (*env)->ReleaseDoubleArrayElements(env, alpha, al, JNI_ABORT);
    (*env)->ReleaseIntArrayElements(env, devices, dev, JNI_ABORT);
    if (rc) { throw_last(env, NULL); return 0; }
    return (jlong)(intptr_t)h;
}

JNIEXPORT void JNICALL CLS(setPhiSampler)(JNIEnv *env, jclass c, jlong h, jint sampler, jint aliasPoissonThreshold)
{
    (void)c;
    if (ldagpu_set_phi_sampler((ldagpu_handle)(intptr_t)h, sampler, aliasPoissonThreshold))
        throw_last(env, (ldagpu_handle)(intptr_t)h);
}

JNIEXPORT void JNICALL CLS(destroy)(JNIEnv *env, jclass c, jlong h)
{
    (void)env; (void)c;
    ldagpu_destroy((ldagpu_handle)(intptr_t)h);
}

JNIEXPORT void JNICALL CLS(initZJavaRandom)(JNIEnv *env, jclass c, jlong h, jint seed)
{
    (void)c;
    if (ldagpu_init_z_java_random((ldagpu_handle)(intptr_t)h, seed)) throw_last(env, (ldagpu_handle)(intptr_t)h);
}

/* sample(iterations) + the copy of z back into the documents' LabelSequences (one call, copy overlapped) */
JNIEXPORT jint JNICALL CLS(sweepGetZ)(JNIEnv *env, jclass c, jlong h, jint n, jintArray z)
{
    (void)c;
    int32_t done = 0;
    jint *zp = (*env)->GetIntArrayElements(env, z, NULL);
    int rc = ldagpu_sweep_get_z((ldagpu_handle)(intptr_t)h, n, &done, (int32_t *)zp);
    (*env)->ReleaseIntArrayElements(env, z, zp, rc ? JNI_ABORT : 0);
    if (rc) throw_last(env, (ldagpu_handle)(intptr_t)h);
    return done;
}

JNIEXPORT void JNICALL CLS(setZ)(JNIEnv *env, jclass c, jlong h, jintArray z, jboolean redrawPhi)
{
    (void)c;
    jint *zp = (*env)->GetIntArrayElements(env, z, NULL);
    int rc = ldagpu_set_z((ldagpu_handle)(intptr_t)h, (const int32_t *)zp, redrawPhi ? 1 : 0);
    (*env)->ReleaseIntArrayElements(env, z, zp, JNI_ABORT);
    if (rc) throw_last(env, (ldagpu_handle)(intptr_t)h);
}

#define GETTER(jname, cfn, jarr, jelem, ctype, Get, Release)                                    \
    JNIEXPORT void JNICALL CLS(jname)(JNIEnv *env, jclass c, jlong h, jarr out)                  \
    {                                                                                            \
        (void)c;                                                                                 \
        jelem *p = (*env)->Get(env, out, NULL);                                                  \
        int rc = cfn((ldagpu_handle)(intptr_t)h, (ctype *)p);                                    \
        (*env)->Release(env, out, p, rc ? JNI_ABORT : 0);                                        \
        if (rc) throw_last(env, (ldagpu_handle)(intptr_t)h);                                     \
    }
GETTER(getTypeTopicCounts, ldagpu_get_type_topic_counts, jintArray, jint, int32_t, GetIntArrayElements, ReleaseIntArrayElements)
GETTER(getTopicTotals, ldagpu_get_topic_totals, jintArray, jint, int32_t, GetIntArrayElements, ReleaseIntArrayElements)
GETTER(getPhi, ldagpu_get_phi, jdoubleArray, jdouble, double, GetDoubleArrayElements, ReleaseDoubleArrayElements)

JNIEXPORT jdouble JNICALL CLS(logLikelihood)(JNIEnv *env, jclass c, jlong h)
{
    (void)c;
    double v = 0.0;
    if (ldagpu_log_likelihood((ldagpu_handle)(intptr_t)h, &v)) throw_last(env, (ldagpu_handle)(intptr_t)h);
    return v;
}

JNIEXPORT jdouble JNICALL CLS(logPosterior)(JNIEnv *env, jclass c, jlong h)
{
    (void)c;
    double v = 0.0;
    if (ldagpu_log_posterior((ldagpu_handle)(intptr_t)h, &v)) throw_last(env, (ldagpu_handle)(intptr_t)h);
    return v;
}

JNIEXPORT void JNICALL CLS(abort)(JNIEnv *env, jclass c, jlong h)
{
    (void)env; (void)c;
    ldagpu_abort((ldagpu_handle)(intptr_t)h);
}

/* hyper-parameter optimisation hooks (ModifiedSimpleLDA.java:812-905): MALLET's fixed point stays in Java */
JNIEXPORT void JNICALL CLS(getCountHistograms)(JNIEnv *env, jclass c, jlong h, jlongArray docTopicHist,
                                               jlongArray typeTopicHist)
{
    (void)c;
    jsize nd = (*env)->GetArrayLength(env, docTopicHist), nt = (*env)->GetArrayLength(env, typeTopicHist);
    jlong *d = (*env)->GetLongArrayElements(env, docTopicHist, NULL);
    jlong *t = (*env)->GetLongArrayElements(env, typeTopicHist, NULL);
    int rc = ldagpu_get_count_histograms((ldagpu_handle)(intptr_t)h, (int32_t)nd, nd ? (int64_t *)d : NULL,
                                         (int32_t)nt, nt ? (int64_t *)t : NULL);
    (*env)->ReleaseLongArrayElements(env, docTopicHist, d, 0);
    (*env)->ReleaseLongArrayElements(env, typeTopicHist, t, 0);
    if (rc) throw_last(env, (ldagpu_handle)(intptr_t)h);
}

JNIEXPORT void JNICALL CLS(setAlpha)(JNIEnv *env, jclass c, jlong h, jdoubleArray alpha)
{
    (void)c;
    jdouble *a = (*env)->GetDoubleArrayElements(env, alpha, NULL);
    int rc = ldagpu_set_alpha((ldagpu_handle)(intptr_t)h, (const double *)a);
    (*env)->ReleaseDoubleArrayElements(env, alpha, a, JNI_ABORT);
    if (rc) throw_last(env, (ldagpu_handle)(intptr_t)h);
}

JNIEXPORT void JNICALL CLS(setBeta)(JNIEnv *env, jclass c, jlong h, jdouble beta)
{
    (void)c;
    if (ldagpu_set_beta((ldagpu_handle)(intptr_t)h, beta)) throw_last(env, (ldagpu_handle)(intptr_t)h);
}

JNIEXPORT void JNICALL CLS(setTestDocuments)(JNIEnv *env, jclass c, jlong h, jlongArray docOffsets, jintArray tokens)
{
    (void)c;
    const jsize D = (*env)->GetArrayLength(env, docOffsets) - 1;
    jlong *off = (*env)->GetLongArrayElements(env, docOffsets, NULL);
    jint *tok = (*env)->GetIntArrayElements(env, tokens, NULL);
    const int rc = ldagpu_set_test_documents((ldagpu_handle)(intptr_t)h, D > 0 ? D : 0, (const int64_t *)off,
                                             (const int32_t *)tok, 0, 0);
    (*env)->ReleaseLongArrayElements(env, docOffsets, off, JNI_ABORT);
    (*env)->ReleaseIntArrayElements(env, tokens, tok, JNI_ABORT);
    if (rc) throw_last(env, (ldagpu_handle)(intptr_t)h);
}

JNIEXPORT jdouble JNICALL CLS(heldOutLogLikelihood)(JNIEnv *env, jclass c, jlong h, jint nParticles)
{
    (void)c;
    double v = 0.0;
    if (ldagpu_heldout_log_likelihood((ldagpu_handle)(intptr_t)h, nParticles, NULL, &v)) throw_last(env, (ldagpu_handle)(intptr_t)h);
    return v;
}
