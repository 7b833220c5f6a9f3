/*
 * mvsim_jni.c -- JNI stubs of net.preibisch.simulation.gpu.Mvsim (java/net/preibisch/simulation/gpu/Mvsim.java):
 * one function per native method, each a direct call into the C ABI of libmvsim.so (include/mvsim.h).
 *
 *     cc -shared -fPIC -I$JAVA_HOME/include -I$JAVA_HOME/include/linux -Iinclude jni/mvsim_jni.c \
 *        -Lmultiview-simulation_b200 -lmvsim -o libmvsim_jni.so
 *
 * Buffers are direct java.nio buffers over pinned host memory (mvsim_alloc_pinned); the stubs check their capacity
 * against the dims before the call, so a wrong shape surfaces as MVSIM_EINVAL instead of a wild read.  No JDK exists in
 * the build image of this repository: tests/test_java_boundary.py compiles this file against a stand-in jni.h and links
 * it against libmvsim.so to prove that names, arities and types match the header.
 */
#include <jni.h>
#include <stdint.h>
#include <string.h>

#include "mvsim.h"

#define MVSIM_JNI(ret, name) JNIEXPORT ret JNICALL Java_net_preibisch_simulation_gpu_Mvsim_##name
#define MAX_VIEWS 64

static mvsim_ctx* ctx_of(jlong h) { return (mvsim_ctx*)(intptr_t)h; }

/* direct buffer address when it holds at least `need` floats, else NULL */
static float* floats_of(JNIEnv* env, jobject buf, int64_t need)
{
    if (!buf) return NULL;
    float* p = (float*)(*env)->GetDirectBufferAddress(env, buf);
    const jlong cap = (*env)->GetDirectBufferCapacity(env, buf);      /* in elements of the buffer's type */
    if (!p || cap < need) return NULL;
    return p;
}

static int dims_of(JNIEnv* env, jlongArray arr, int64_t d[3])
{
    if (!arr || (*env)->GetArrayLength(env, arr) < 3) return MVSIM_EINVAL;
    jlong tmp[3];
    (*env)->GetLongArrayRegion(env, arr, 0, 3, tmp);
    for (int i = 0; i < 3; ++i) {
        if (tmp[i] < 1) return MVSIM_EINVAL;
        d[i] = (int64_t)tmp[i];
    }
    return MVSIM_OK;
}

static int64_t prod3(const int64_t d[3]) { return d[0] * d[1] * d[2]; }
static int64_t slices_of(const int64_t d[3], int inc) { return d[0] * d[1] * ((d[2] - 1) / inc + 1); }

/* ---- library / context ------------------------------------------------------------------------------------------- */
MVSIM_JNI(jint, version)(JNIEnv* env, jclass c)
{
    (void)env; (void)c;
    return mvsim_version();
}

MVSIM_JNI(jint, deviceCount)(JNIEnv* env, jclass c)
{
    (void)env; (void)c;
    int n = 0;
    return mvsim_device_count(&n) == MVSIM_OK ? n : -1;
}

MVSIM_JNI(jlong, ctxCreate)(JNIEnv* env, jclass c, jint device)
{
    (void)env; (void)c;
    mvsim_ctx* ctx = NULL;
    if (mvsim_ctx_create(device, &ctx) != MVSIM_OK) return 0;
    return (jlong)(intptr_t)ctx;
}

MVSIM_JNI(void, ctxDestroy)(JNIEnv* env, jclass c, jlong ctx)
{
    (void)env; (void)c;
    mvsim_ctx_destroy(ctx_of(ctx));
}

MVSIM_JNI(jint, ctxSynchronize)(JNIEnv* env, jclass c, jlong ctx)
{
    (void)env; (void)c;
    return mvsim_ctx_synchronize(ctx_of(ctx));
}

MVSIM_JNI(jstring, lastError)(JNIEnv* env, jclass c, jlong ctx)
{
    (void)c;
    const char* msg = mvsim_last_error(ctx_of(ctx));
    return (*env)->NewStringUTF(env, msg ? msg : "");
}

MVSIM_JNI(jobject, allocPinned)(JNIEnv* env, jclass c, jlong bytes)
{
    (void)c;
    void* p = NULL;
    if (bytes < 0 || mvsim_alloc_pinned((size_t)bytes, &p) != MVSIM_OK) return NULL;
    jobject buf = (*env)->NewDirectByteBuffer(env, p, bytes);
    if (!buf) mvsim_free_pinned(p);
    return buf;
}

MVSIM_JNI(void, freePinned)(JNIEnv* env, jclass c, jobject buffer)
{
    (void)c;
    if (buffer) mvsim_free_pinned((*env)->GetDirectBufferAddress(env, buffer));
}

MVSIM_JNI(jint, convPaddedDims)(JNIEnv* env, jclass c, jlongArray dims, jlongArray kdims, jlongArray nfft_out)
{
    (void)c;
    int64_t d[3], k[3], n[3];
    if (dims_of(env, dims, d) || dims_of(env, kdims, k) || !nfft_out || (*env)->GetArrayLength(env, nfft_out) < 3) return MVSIM_EINVAL;
    const int st = mvsim_conv_padded_dims(d, k, n);
    if (st == MVSIM_OK) {
        const jlong out[3] = { (jlong)n[0], (jlong)n[1], (jlong)n[2] };
        (*env)->SetLongArrayRegion(env, nfft_out, 0, 3, out);
    }
    return st;
}

MVSIM_JNI(jint, ctxSetOption)(JNIEnv* env, jclass c, jlong ctx, jint option, jlong value)
{
    (void)env; (void)c;
    return mvsim_ctx_set_option(ctx_of(ctx), option, (int64_t)value);
}

MVSIM_JNI(jint, psfCacheConfigure)(JNIEnv* env, jclass c, jlong ctx, jlong max_bytes)
{
    (void)env; (void)c;
    if (max_bytes < 0) return MVSIM_EINVAL;
    return mvsim_psf_cache_configure(ctx_of(ctx), (size_t)max_bytes);
}

MVSIM_JNI(jint, psfCacheStats)(JNIEnv* env, jclass c, jlong ctx, jlongArray stats4)
{
    (void)c;
    if (!stats4 || (*env)->GetArrayLength(env, stats4) < 4) return MVSIM_EINVAL;
    int64_t st[4];
    const int rc = mvsim_psf_cache_stats(ctx_of(ctx), st);
    if (rc == MVSIM_OK) {
        const jlong out[4] = { (jlong)st[0], (jlong)st[1], (jlong)st[2], (jlong)st[3] };
        (*env)->SetLongArrayRegion(env, stats4, 0, 4, out);
    }
    return rc;
}

/* ---- stage entry points -------------------------------------------------------------------------------------------- */
MVSIM_JNI(jint, axisRotation)(JNIEnv* env, jclass c, jlongArray dims, jint axis, jint degrees, jdoubleArray fwd12, jdoubleArray inv12)
{
    (void)c;
    int64_t d[3];
    double fwd[12], inv[12];
    if (dims_of(env, dims, d)) return MVSIM_EINVAL;
    const int st = mvsim_axis_rotation(d, axis, degrees, fwd, inv);
    if (st != MVSIM_OK) return st;
    if (fwd12 && (*env)->GetArrayLength(env, fwd12) >= 12) (*env)->SetDoubleArrayRegion(env, fwd12, 0, 12, fwd);
    if (inv12 && (*env)->GetArrayLength(env, inv12) >= 12) (*env)->SetDoubleArrayRegion(env, inv12, 0, 12, inv);
    return MVSIM_OK;
}

MVSIM_JNI(jint, rotateAxis)(JNIEnv* env, jclass c, jlong ctx, jobject in, jobject out, jlongArray dims, jint axis, jint degrees)
{
    (void)c;
    int64_t d[3];
    if (dims_of(env, dims, d)) return MVSIM_EINVAL;
    const float* src = floats_of(env, in, prod3(d));
    float* dst = floats_of(env, out, prod3(d));
    if (!src || !dst) return MVSIM_EINVAL;
    return mvsim_rotate_axis(ctx_of(ctx), src, dst, d, axis, degrees);
}

MVSIM_JNI(jint, attenuate)(JNIEnv* env, jclass c, jlong ctx, jobject in, jobject out, jlongArray dims, jdouble delta, jboolean strict)
{
    (void)c;
    int64_t d[3];
    if (dims_of(env, dims, d)) return MVSIM_EINVAL;
    const float* src = floats_of(env, in, prod3(d));
    float* dst = floats_of(env, out, prod3(d));
    if (!src || !dst) return MVSIM_EINVAL;
    return mvsim_attenuate(ctx_of(ctx), src, dst, d, delta, strict ? 1 : 0);
}

MVSIM_JNI(jint, psfNormalize)(JNIEnv* env, jclass c, jlong ctx, jobject psf, jlongArray kdims, jdoubleArray sum_out)
{
    (void)c;
    int64_t k[3];
    if (dims_of(env, kdims, k)) return MVSIM_EINVAL;
    float* p = floats_of(env, psf, prod3(k));
    if (!p) return MVSIM_EINVAL;
    double sum = 0.0;
    const int st = mvsim_psf_normalize(ctx_of(ctx), p, k, &sum);
    if (st == MVSIM_OK && sum_out && (*env)->GetArrayLength(env, sum_out) >= 1) (*env)->SetDoubleArrayRegion(env, sum_out, 0, 1, &sum);
    return st;
}

MVSIM_JNI(jint, convolve)(JNIEnv* env, jclass c, jlong ctx, jobject img, jlongArray dims, jobject psf, jlongArray kdims, jobject out)
{
    (void)c;
    int64_t d[3], k[3];
    if (dims_of(env, dims, d) || dims_of(env, kdims, k)) return MVSIM_EINVAL;
    const float* src = floats_of(env, img, prod3(d));
    float* kern = floats_of(env, psf, prod3(k));
    float* dst = floats_of(env, out, prod3(d));
    if (!src || !kern || !dst) return MVSIM_EINVAL;
    return mvsim_convolve(ctx_of(ctx), src, d, kern, k, dst);
}

MVSIM_JNI(jint, adjust)(JNIEnv* env, jclass c, jlong ctx, jobject img, jlongArray dims, jfloat min_value, jfloat target_avg, jdoubleArray corr_out)
{
    (void)c;
    int64_t d[3];
    if (dims_of(env, dims, d)) return MVSIM_EINVAL;
    float* p = floats_of(env, img, prod3(d));
    if (!p) return MVSIM_EINVAL;
    double corr = 0.0;
    const int st = mvsim_adjust(ctx_of(ctx), p, d, min_value, target_avg, &corr);
    if (st == MVSIM_OK && corr_out && (*env)->GetArrayLength(env, corr_out) >= 1) (*env)->SetDoubleArrayRegion(env, corr_out, 0, 1, &corr);
    return st;
}

MVSIM_JNI(jint, extractSlices)(JNIEnv* env, jclass c, jlong ctx, jobject in, jlongArray dims, jint inc, jfloat snr, jlong seed, jlong stream, jobject out)
{
    (void)c;
    int64_t d[3];
    if (dims_of(env, dims, d) || inc < 1) return MVSIM_EINVAL;
    const float* src = floats_of(env, in, prod3(d));
    float* dst = floats_of(env, out, slices_of(d, inc));
    if (!src || !dst) return MVSIM_EINVAL;
    return mvsim_extract_slices(ctx_of(ctx), src, d, inc, snr, (uint64_t)seed, (uint64_t)stream, dst);
}

MVSIM_JNI(jint, poisson)(JNIEnv* env, jclass c, jlong ctx, jobject inout, jlong n, jdouble snr, jlong seed, jlong stream)
{
    (void)c;
    if (n < 0) return MVSIM_EINVAL;
    float* p = floats_of(env, inout, n);
    if (!p && n > 0) return MVSIM_EINVAL;
    return mvsim_poisson(ctx_of(ctx), p, (size_t)n, snr, (uint64_t)seed, (uint64_t)stream);
}

static void fill_params(mvsim_view_params* p, const int64_t d[3], const int64_t k[3], jint axis, jint degrees, jdouble delta, jfloat min_value,
                        jfloat target_avg, jint inc, jfloat snr, jlong seed, jlong stream, jboolean strict)
{
    memset(p, 0, sizeof(*p));
    for (int i = 0; i < 3; ++i) { p->dims[i] = d[i]; p->kdims[i] = k[i]; }
    p->axis = axis; p->degrees = degrees; p->delta = delta;
    p->min_value = min_value; p->target_avg = target_avg;
    p->inc = inc; p->snr = snr;
    p->seed = (uint64_t)seed; p->stream = (uint64_t)stream;
    p->strict_reference = strict ? 1 : 0;
}

MVSIM_JNI(jint, simulateView)(JNIEnv* env, jclass c, jlong ctx, jlongArray dims, jlongArray kdims, jint axis, jint degrees, jdouble delta,
                              jfloat min_value, jfloat target_avg, jint inc, jfloat snr, jlong seed, jlong stream, jboolean strict,
                              jobject gt, jobject psf, jobject out)
{
    (void)c;
    int64_t d[3], k[3];
    if (dims_of(env, dims, d) || dims_of(env, kdims, k) || inc < 1) return MVSIM_EINVAL;
    const float* src = floats_of(env, gt, prod3(d));
    float* kern = floats_of(env, psf, prod3(k));
    float* dst = floats_of(env, out, slices_of(d, inc));
    if (!src || !kern || !dst) return MVSIM_EINVAL;
    mvsim_view_params p;
    fill_params(&p, d, k, axis, degrees, delta, min_value, target_avg, inc, snr, seed, stream, strict);
    return mvsim_simulate_view(ctx_of(ctx), &p, src, kern, dst);
}

MVSIM_JNI(jint, simulateViews)(JNIEnv* env, jclass c, jlong ctx, jlongArray dims, jlongArray kdims, jint axis, jintArray degrees, jdouble delta,
                               jfloat min_value, jfloat target_avg, jint inc, jfloat snr, jlong seed, jlong first_stream, jboolean strict,
                               jobject gt, jobjectArray psfs, jobjectArray outs)
{
    (void)c;
    int64_t d[3], k[3];
    if (dims_of(env, dims, d) || dims_of(env, kdims, k) || inc < 1 || !degrees || !psfs || !outs) return MVSIM_EINVAL;
    const jsize n = (*env)->GetArrayLength(env, degrees);
    if (n < 0 || n > MAX_VIEWS || (*env)->GetArrayLength(env, psfs) < n || (*env)->GetArrayLength(env, outs) < n) return MVSIM_EINVAL;
    const float* src = floats_of(env, gt, prod3(d));
    if (!src) return MVSIM_EINVAL;
    jint deg[MAX_VIEWS];
    (*env)->GetIntArrayRegion(env, degrees, 0, n, deg);
    mvsim_view_params params[MAX_VIEWS];
    float* kern[MAX_VIEWS];
    float* dst[MAX_VIEWS];
    for (jsize v = 0; v < n; ++v) {
        kern[v] = floats_of(env, (*env)->GetObjectArrayElement(env, psfs, v), prod3(k));
        dst[v] = floats_of(env, (*env)->GetObjectArrayElement(env, outs, v), slices_of(d, inc));
        if (!kern[v] || !dst[v]) return MVSIM_EINVAL;
        fill_params(&params[v], d, k, axis, deg[v], delta, min_value, target_avg, inc, snr, seed, first_stream + v, strict);
    }
    return mvsim_simulate_views(ctx_of(ctx), (int)n, params, src, kern, dst);
}

/* element i of an optional array of output buffers: NULL when the array or the element is null; *bad when it is too small */
static float* opt_floats_of(JNIEnv* env, jobjectArray arr, jsize i, int64_t need, int* bad)
{
    if (!arr) return NULL;
    if ((*env)->GetArrayLength(env, arr) <= i) { *bad = 1; return NULL; }
    jobject b = (*env)->GetObjectArrayElement(env, arr, i);
    if (!b) return NULL;
    float* p = floats_of(env, b, need);
    if (!p) *bad = 1;
    return p;
}

MVSIM_JNI(jint, simulateDataset)(JNIEnv* env, jclass c, jlong ctx, jlongArray dims, jlongArray kdims, jintArray degrees, jintArray align_degrees,
                                 jdouble delta, jfloat min_value, jfloat target_avg, jint inc, jfloat snr, jlongArray seeds, jboolean strict,
                                 jfloat osem, jintArray views, jobject gt, jobjectArray psfs, jobjectArray acq, jobjectArray aligned,
                                 jobjectArray aligned_psf, jobjectArray weights, jobject sum_weights)
{
    (void)c;
    int64_t d[3], k[3];
    if (dims_of(env, dims, d) || dims_of(env, kdims, k) || inc < 1 || !degrees || !align_degrees || !seeds || !views || !psfs) return MVSIM_EINVAL;
    const jsize n_all = (*env)->GetArrayLength(env, degrees), n = (*env)->GetArrayLength(env, views);
    if (n_all < 1 || n_all > MVSIM_MAX_WEIGHT_VIEWS || (*env)->GetArrayLength(env, align_degrees) < n_all ||
        (*env)->GetArrayLength(env, seeds) < n_all || n > n_all || (*env)->GetArrayLength(env, psfs) < n)
        return MVSIM_EINVAL;
    const float* src = floats_of(env, gt, prod3(d));
    if (!src) return MVSIM_EINVAL;
    jint deg[MVSIM_MAX_WEIGHT_VIEWS], adeg[MVSIM_MAX_WEIGHT_VIEWS], vw[MVSIM_MAX_WEIGHT_VIEWS];
    jlong sd[MVSIM_MAX_WEIGHT_VIEWS];
    (*env)->GetIntArrayRegion(env, degrees, 0, n_all, deg);
    (*env)->GetIntArrayRegion(env, align_degrees, 0, n_all, adeg);
    (*env)->GetLongArrayRegion(env, seeds, 0, n_all, sd);
    (*env)->GetIntArrayRegion(env, views, 0, n, vw);
    mvsim_view_params params[MVSIM_MAX_WEIGHT_VIEWS];
    int32_t align[MVSIM_MAX_WEIGHT_VIEWS], sel[MVSIM_MAX_WEIGHT_VIEWS];
    for (jsize v = 0; v < n_all; ++v) {
        fill_params(&params[v], d, k, 0, deg[v], delta, min_value, target_avg, inc, snr, sd[v], v, strict);
        align[v] = adeg[v];
    }
    const int64_t aligned_elems = d[0] * d[1] * (((d[2] - 1) / inc) * inc + 1);
    float* kern[MVSIM_MAX_WEIGHT_VIEWS];
    mvsim_dataset_outputs outs[MVSIM_MAX_WEIGHT_VIEWS];
    int bad = 0;
    for (jsize i = 0; i < n; ++i) {
        sel[i] = vw[i];
        kern[i] = floats_of(env, (*env)->GetObjectArrayElement(env, psfs, i), prod3(k));
        if (!kern[i]) return MVSIM_EINVAL;
        outs[i].acq = opt_floats_of(env, acq, i, slices_of(d, inc), &bad);
        outs[i].aligned = opt_floats_of(env, aligned, i, aligned_elems, &bad);
        outs[i].aligned_psf = opt_floats_of(env, aligned_psf, i, prod3(k), &bad);
        outs[i].weights = opt_floats_of(env, weights, i, prod3(d), &bad);
    }
    float* sum = sum_weights ? floats_of(env, sum_weights, prod3(d)) : NULL;
    if (bad || (sum_weights && !sum)) return MVSIM_EINVAL;
    return mvsim_simulate_dataset(ctx_of(ctx), (int)n_all, params, align, osem, (int)n, sel, src, kern, outs, sum);
}

/* ---- post-acquisition chain ------------------------------------------------------------------------------------------ */
MVSIM_JNI(jint, makeIsotropic)(JNIEnv* env, jclass c, jlong ctx, jobject in, jlongArray dims, jint inc, jobject out)
{
    (void)c;
    int64_t d[3];
    if (dims_of(env, dims, d) || inc < 1) return MVSIM_EINVAL;
    const float* src = floats_of(env, in, prod3(d));
    float* dst = floats_of(env, out, d[0] * d[1] * ((d[2] - 1) * inc + 1));
    if (!src || !dst) return MVSIM_EINVAL;
    return mvsim_make_isotropic(ctx_of(ctx), src, d, inc, dst);
}

MVSIM_JNI(jint, weightImage)(JNIEnv* env, jclass c, jlong ctx, jlongArray dims, jobject out)
{
    (void)c;
    int64_t d[3];
    if (dims_of(env, dims, d)) return MVSIM_EINVAL;
    float* dst = floats_of(env, out, prod3(d));
    if (!dst) return MVSIM_EINVAL;
    return mvsim_weight_image(ctx_of(ctx), d, dst);
}

MVSIM_JNI(jint, normalizeWeights)(JNIEnv* env, jclass c, jlong ctx, jobjectArray weights, jlongArray dims, jfloat osem, jobject sum_out)
{
    (void)c;
    int64_t d[3];
    if (dims_of(env, dims, d) || !weights) return MVSIM_EINVAL;
    const jsize n = (*env)->GetArrayLength(env, weights);
    if (n < 1 || n > MVSIM_MAX_WEIGHT_VIEWS) return MVSIM_EINVAL;
    float* w[MVSIM_MAX_WEIGHT_VIEWS];
    for (jsize v = 0; v < n; ++v) {
        w[v] = floats_of(env, (*env)->GetObjectArrayElement(env, weights, v), prod3(d));
        if (!w[v]) return MVSIM_EINVAL;
    }
    float* sum = sum_out ? floats_of(env, sum_out, prod3(d)) : NULL;
    if (sum_out && !sum) return MVSIM_EINVAL;
    return mvsim_normalize_weights(ctx_of(ctx), w, (int)n, d, osem, sum);
}

/* ---- device-resident volumes ---------------------------------------------------------------------------------------- */
static mvsim_volume* vol_of(jlong h) { return (mvsim_volume*)(intptr_t)h; }

/* direct buffer address when it holds the whole volume, else NULL */
static float* volume_floats_of(JNIEnv* env, jlong vol, jobject buf)
{
    int64_t d[3];
    if (!vol || mvsim_volume_dims(vol_of(vol), d) != MVSIM_OK) return NULL;
    return floats_of(env, buf, prod3(d));
}

/* three longs, any sign (interval bounds: the library checks them against the volume) */
static int longs3_of(JNIEnv* env, jlongArray arr, int64_t v[3])
{
    if (!arr || (*env)->GetArrayLength(env, arr) < 3) return MVSIM_EINVAL;
    jlong tmp[3];
    (*env)->GetLongArrayRegion(env, arr, 0, 3, tmp);
    for (int i = 0; i < 3; ++i) v[i] = (int64_t)tmp[i];
    return MVSIM_OK;
}

MVSIM_JNI(jlong, volumeCreate)(JNIEnv* env, jclass c, jlong ctx, jlongArray dims)
{
    (void)c;
    int64_t d[3];
    mvsim_volume* v = NULL;
    if (dims_of(env, dims, d) || mvsim_volume_create(ctx_of(ctx), d, &v) != MVSIM_OK) return 0;
    return (jlong)(intptr_t)v;
}

MVSIM_JNI(jint, volumeFree)(JNIEnv* env, jclass c, jlong ctx, jlong vol)
{
    (void)env; (void)c;
    return mvsim_volume_free(ctx_of(ctx), vol_of(vol));
}

MVSIM_JNI(jint, volumeUpload)(JNIEnv* env, jclass c, jlong ctx, jlong vol, jobject host)
{
    (void)c;
    const float* src = volume_floats_of(env, vol, host);
    if (!src) return MVSIM_EINVAL;
    return mvsim_volume_upload(ctx_of(ctx), vol_of(vol), src);
}

MVSIM_JNI(jint, volumeDownload)(JNIEnv* env, jclass c, jlong ctx, jlong vol, jobject host)
{
    (void)c;
    float* dst = volume_floats_of(env, vol, host);
    if (!dst) return MVSIM_EINVAL;
    return mvsim_volume_download(ctx_of(ctx), vol_of(vol), dst);
}

MVSIM_JNI(jint, devSimulatePhantom)(JNIEnv* env, jclass c, jlong ctx, jint size, jboolean half, jlong seed, jlong out, jlongArray n_small_out)
{
    (void)c;
    int64_t n = 0;
    const int st = mvsim_dev_simulate_phantom(ctx_of(ctx), size, half ? 1 : 0, (int64_t)seed, vol_of(out), &n);
    if (st == MVSIM_OK && n_small_out && (*env)->GetArrayLength(env, n_small_out) >= 1) {
        const jlong v = (jlong)n;
        (*env)->SetLongArrayRegion(env, n_small_out, 0, 1, &v);
    }
    return st;
}

MVSIM_JNI(jint, devPsfNormalize)(JNIEnv* env, jclass c, jlong ctx, jlong psf, jdoubleArray sum_out)
{
    (void)c;
    double sum = 0.0;
    const int st = mvsim_dev_psf_normalize(ctx_of(ctx), vol_of(psf), sum_out ? &sum : NULL);
    if (st == MVSIM_OK && sum_out && (*env)->GetArrayLength(env, sum_out) >= 1) (*env)->SetDoubleArrayRegion(env, sum_out, 0, 1, &sum);
    return st;
}

MVSIM_JNI(jint, devAttenuate)(JNIEnv* env, jclass c, jlong ctx, jlong in, jlong out, jdouble delta, jboolean strict)
{
    (void)env; (void)c;
    return mvsim_dev_attenuate(ctx_of(ctx), vol_of(in), vol_of(out), delta, strict ? 1 : 0);
}

MVSIM_JNI(jint, devConvolve)(JNIEnv* env, jclass c, jlong ctx, jlong img, jlong psf, jlong out)
{
    (void)env; (void)c;
    return mvsim_dev_convolve(ctx_of(ctx), vol_of(img), vol_of(psf), vol_of(out));
}

MVSIM_JNI(jint, devAdjust)(JNIEnv* env, jclass c, jlong ctx, jlong img, jfloat min_value, jfloat target_avg, jdoubleArray corr_out)
{
    (void)c;
    double corr = 0.0;
    const int st = mvsim_dev_adjust(ctx_of(ctx), vol_of(img), min_value, target_avg, corr_out ? &corr : NULL);
    if (st == MVSIM_OK && corr_out && (*env)->GetArrayLength(env, corr_out) >= 1) (*env)->SetDoubleArrayRegion(env, corr_out, 0, 1, &corr);
    return st;
}

MVSIM_JNI(jint, devExtractInterval)(JNIEnv* env, jclass c, jlong ctx, jlong in, jlongArray min, jlongArray max, jint inc, jfloat snr, jlong seed,
                                    jlong stream, jlong out)
{
    (void)c;
    int64_t mn[3], mx[3];
    if (longs3_of(env, min, mn) || longs3_of(env, max, mx)) return MVSIM_EINVAL;
    return mvsim_dev_extract_interval(ctx_of(ctx), vol_of(in), mn, mx, inc, snr, (uint64_t)seed, (uint64_t)stream, vol_of(out));
}
