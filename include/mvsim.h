/*
 * mvsim.h -- C ABI of libmvsim.so: the B200 (sm_100a) implementation of the per-view acquisition
 * pipeline of PreibischLab/multiview-simulation.
 *
 * The reference has no FFI layer; its boundary for this path is a set of public static Java
 * methods (S = src/main/java/net/preibisch/simulation):
 *     S/SimulateMultiViewDataset.java:80   axisRotation
 *     S/SimulateMultiViewDataset.java:104  rotateAroundAxis
 *     S/SimulateMultiViewDataset.java:318  attenuate3d
 *     S/SimulateMultiViewDataset.java:253  convolve            (+ S/Tools.java:112 normImage)
 *     S/Tools.java:143                     adjustImage
 *     S/SimulateMultiViewDataset.java:195  extractSlices
 *     S/SimulateMultiViewDataset.java:233  poissonProcess      (+ S/Tools.java:73)
 * Each entry point below names the method whose body it replaces; INTEGRATION.md shows the JNI /
 * Panama stubs a maintainer adds on the Java side.
 *
 * Conventions
 *   - volumes are dense float32 in ImgLib2 ArrayImg order, x fastest: idx = x + X*(y + Y*z);
 *     dims[3] = {X, Y, Z}.
 *   - every function returns an mvsim_status (0 = OK); mvsim_last_error(ctx) has the text.
 *   - host entry points (const float* / float* arguments) copy to the device, run the CUDA
 *     kernels and copy back; they return after the result is in the caller's buffer.  Buffers from
 *     mvsim_alloc_pinned make the copies asynchronous DMA.
 *   - device entry points (mvsim_volume handles) keep data resident in HBM between stages and are
 *     asynchronous on the context's stream.
 *   - one context = one device + one stream + cached workspaces.  A context must not be used from
 *     two threads at once; any number of contexts may exist per device (the reference's callers
 *     run two pipelines concurrently, S/SimulateTileStitching.java:85-117).
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     MVSIM_ECUDA.
 */
#ifndef MVSIM_H
#define MVSIM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum mvsim_status {
    MVSIM_OK = 0,
    MVSIM_EINVAL = 1,       /* bad argument / shape (the reference throws from imglib2) */
    MVSIM_ENOMEM = 2,
    MVSIM_ECUDA = 3,
    MVSIM_ENCCL = 4,
    MVSIM_EUNSUPPORTED = 5  /* padded size beyond the FFT size table */
} mvsim_status;

typedef struct mvsim_ctx mvsim_ctx;
typedef struct mvsim_volume mvsim_volume;   /* device-resident float32 volume */

/* Parameters of one view: loop body S/SimulateMultiViewDataset.java:570-585. */
typedef struct mvsim_view_params {
    int64_t dims[3];        /* ground-truth volume X, Y, Z */
    int64_t kdims[3];       /* PSF KX, KY, KZ */
    int32_t axis;           /* rotation axis (reference uses 0) */
    int32_t degrees;        /* angle + angleOffset, integer degrees (:570) */
    double delta;           /* attenuation (:573), reference 0.01 */
    float min_value;        /* adjustImage minValue (:77), 0.0001f */
    float target_avg;       /* adjustImage targetAverage (:78), 1 */
    int32_t inc;            /* lightsheetSpacing (:585) */
    float snr;              /* poissonSNR; < 0 = no noise (:211) */
    uint64_t seed;          /* Philox key; the Java facade draws it from the caller's Random */
    uint64_t stream;        /* Philox stream id = view id */
    int32_t strict_reference; /* 1: attenuate loops dimension(0) steps like :345 (needs X <= Y) */
    int32_t reserved;
} mvsim_view_params;

/* stage indices of mvsim_stage_times */
enum {
    MVSIM_T_H2D = 0, MVSIM_T_ROTATE, MVSIM_T_ATTENUATE, MVSIM_T_PSF, MVSIM_T_FFT_XFWD, MVSIM_T_FFT_YFWD,
    MVSIM_T_FFT_ZFUSED, MVSIM_T_FFT_YINV, MVSIM_T_FFT_XINV, MVSIM_T_ADJUST, MVSIM_T_SAMPLE, MVSIM_T_D2H,
    MVSIM_T_WIDEN,          /* host: uint16 counts -> float32 (count transport), wall-clock milliseconds of the widening threads */
    MVSIM_NSTAGES
};

/* context options (mvsim_ctx_set_option) */
enum {
    /* 1: in the batch calls (mvsim_simulate_views / mvsim_dev_simulate_views) the Poisson counts of a view (snr >= 0) cross the host
     * link as uint16 -- half the device->host bytes, which bound the end-to-end rate -- and are widened to the float32 of the
     * reference's API (Img<FloatType>) by host threads inside the call, overlapped with the later views.  Results are bit-identical to
     * the float32 transport; a view with a count above 65535 is fetched as float32 instead.  0 (default): float32. */
    MVSIM_OPT_COUNT_TRANSPORT = 1,
    /* host threads that widen (0 = default: 4) */
    MVSIM_OPT_HOST_THREADS = 2,
    /* fused z pass of the whole-view calls: 0 (default) = the kernel measured fastest for the shape, 1 = decimated inverse where the
     * split allows it, else full spectral (no polyphase kernel), 2 = full spectral kernel only, 3 = polyphase kernel where the shape
     * allows it.  The variants agree to float32 rounding; the option exists for A/B measurements and cross-checks. */
    MVSIM_OPT_Z_KERNEL = 3
};
int mvsim_ctx_set_option(mvsim_ctx* ctx, int option, int64_t value);

/* ---- library / context ------------------------------------------------------------------- */
int mvsim_version(void);
int mvsim_device_count(int* count);
int mvsim_ctx_create(int device, mvsim_ctx** ctx);
/* same, but all work is enqueued on an existing cudaStream_t (e.g. torch's current stream; NULL = the
 * legacy default stream) */
int mvsim_ctx_create_on_stream(int device, void* cuda_stream, mvsim_ctx** ctx);
int mvsim_ctx_destroy(mvsim_ctx* ctx);
int mvsim_ctx_synchronize(mvsim_ctx* ctx);
const char* mvsim_last_error(mvsim_ctx* ctx);      /* ctx may be NULL: last error of this thread */
/* per-kernel CUDA-event timing: enable, run, then read accumulated milliseconds and launch counts */
int mvsim_profile_enable(mvsim_ctx* ctx, int on);
int mvsim_profile_reset(mvsim_ctx* ctx);
int mvsim_stage_times(mvsim_ctx* ctx, double ms[MVSIM_NSTAGES], int64_t launches[MVSIM_NSTAGES]);
/* number of kernels this context has launched since creation */
int64_t mvsim_kernel_launches(mvsim_ctx* ctx);

/* PSF-spectrum cache of a context (SURVEY C6; OFF by default = the reference's behaviour, which rebuilds the kernel FFT on every
 * call, S/SimulateMultiViewDataset.java:257).  With max_bytes > 0 the convolution keeps the partial spectrum of every distinct
 * (normalised) PSF it has seen, keyed by a 128-bit content hash computed on the device, up to max_bytes of HBM (least recently used
 * out first); repeated PSFs -- SNR sweeps, tile pairs (S/SimulateTileStitching.java:71,95,110), the 8 distinct volumes among the 18
 * fixtures -- then skip the PSF transforms.  Results are bit-identical with and without; the in-place normalisation of the
 * caller's PSF (:255) still happens on every call.  Shrinking the budget drops all entries.
 * stats = { hits, misses, entries, bytes held }. */
int mvsim_psf_cache_configure(mvsim_ctx* ctx, size_t max_bytes);
int mvsim_psf_cache_stats(mvsim_ctx* ctx, int64_t stats[4]);

int mvsim_alloc_pinned(size_t bytes, void** ptr);
int mvsim_free_pinned(void* ptr);

/* FFT padding the convolution will use for (dims, kdims): nfft = {2*Nx/2, Ny, Nz} */
int mvsim_conv_padded_dims(const int64_t dims[3], const int64_t kdims[3], int64_t nfft[3]);

/* ---- host-buffer stage entry points ------------------------------------------------------- */
/* axisRotation (:80-102) and its mpicbg createInverse(); pure host arithmetic, 3x4 row-major */
int mvsim_axis_rotation(const int64_t dims[3], int axis, int degrees, double fwd[12], double inv[12]);
/* rotateAroundAxis (:104-135) */
int mvsim_rotate_axis(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], int axis, int degrees);
/* attenuate3d (:318-364) */
int mvsim_attenuate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], double delta, int strict_reference);
/* Tools.normImage (S/Tools.java:112-118): in place, returns the sum that was divided out */
int mvsim_psf_normalize(mvsim_ctx* ctx, float* psf, const int64_t kdims[3], double* sum_out);
/* convolve (:253-264): normalises psf IN PLACE like :255, then FFT convolution */
int mvsim_convolve(mvsim_ctx* ctx, const float* img, const int64_t dims[3], float* psf, const int64_t kdims[3], float* out);
/* Tools.adjustImage (S/Tools.java:143-159): in place, returns the correction factor */
int mvsim_adjust(mvsim_ctx* ctx, float* img, const int64_t dims[3], float min_value, float target_avg, double* correction_out);
/* extractSlices (:195-231): out has X*Y*((Z-1)/inc+1) floats; snr < 0 copies without noise */
int mvsim_extract_slices(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, float snr,
                         uint64_t seed, uint64_t stream, float* out);
/* Tools.poissonProcess (S/Tools.java:73-86): in place on n floats */
int mvsim_poisson(mvsim_ctx* ctx, float* inout, size_t n, double snr, uint64_t seed, uint64_t stream);
/* whole loop body (:570-585) with intermediates kept on the device.  psf is normalised in place.
 * out has X*Y*((Z-1)/inc+1) floats. */
int mvsim_simulate_view(mvsim_ctx* ctx, const mvsim_view_params* p, const float* gt, float* psf, float* out);

/* the reference's view loop (:567-613): one ground truth, n_views parameter sets / PSFs / outputs.  The
 * ground truth is uploaded once; the download of view v overlaps the kernels of view v+1. */
int mvsim_simulate_views(mvsim_ctx* ctx, int n_views, const mvsim_view_params* params, const float* gt,
                         float* const* psfs, float* const* outs);

/* ---- post-acquisition chain of main() (after the sampler; SURVEY section 8f-1) --------------------------------- */
#define MVSIM_MAX_WEIGHT_VIEWS 16
/* makeIsotropic (:144-171): out has X*Y*((Z-1)*inc+1) floats */
int mvsim_make_isotropic(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, float* out);
/* computeWeightImage (:280-316): cosine taper over 40 px along y (its `delta` argument is unused in the reference) */
int mvsim_weight_image(mvsim_ctx* ctx, const int64_t dims[3], float* out);
/* weight normalisation of main() (:615-661), in place on n_views volumes: w_v = min(1, osem * w_v / sum_v w_v);
 * sum_out (nullable) receives the sum of the normalised weights (sum_weights.tif, :648-663) */
int mvsim_normalize_weights(mvsim_ctx* ctx, float* const* weights, int n_views, const int64_t dims[3], float osem, float* sum_out);

/* main()'s aligned outputs without the intermediate volumes (:588-663).  The dataset calls rotate about x only (main() does); other
 * axes stay with the stage entry points.  mvsim_dev_align_view and mvsim_dev_aligned_weights are declared with the device volumes. */
typedef struct mvsim_dataset_outputs {
    float* acq;             /* X*Y*((Z-1)/inc+1): the acquired view, float32 (MVSIM_OPT_COUNT_TRANSPORT does not apply) */
    float* aligned;         /* X*Y*(((Z-1)/inc)*inc+1): rotateAroundAxis(makeIsotropic(acq, inc), 0, align_degrees) (:588, :591) */
    float* aligned_psf;     /* KX*KY*KZ: the normalised PSF rotated back (:593) */
    float* weights;         /* X*Y*Z: the view's normalised, rotated-back weight image (:576, :592, :615-646) */
} mvsim_dataset_outputs;
/* main()'s view loop with its post-acquisition chain (:567-663) for views[0..n_views) of a dataset of n_all (1..MVSIM_MAX_WEIGHT_VIEWS)
 * views.  params and align_degrees (the rotate-back angles, -angle in main()) describe ALL views: the weight normalisation needs every
 * angle, so any subset of the views -- one rank's share -- gives exactly the volumes of the full set.  psfs[i] and outs[i] belong to
 * views[i]; psfs are normalised in place like :255; any pointer in outs[i] may be NULL (not produced).  sum_weights (nullable):
 * sum_weights.tif (:648-663).  Every params[k].axis must be 0 and all views share the ground truth dims.  The ground truth is
 * uploaded once; at most two views' outputs are held on the device, and the downloads of one view overlap the next view's kernels. */
int mvsim_simulate_dataset(mvsim_ctx* ctx, int n_all, const mvsim_view_params* params, const int32_t* align_degrees, float osem,
                           int n_views, const int32_t* views, const float* gt, float* const* psfs, const mvsim_dataset_outputs* outs,
                           float* sum_weights);

/* ---- input generators either side of the path (SURVEY section 8f rows 2-4) ----------------------------------------
 * java.util.Random is replayed bit-exactly (JDK specification), so the caller's seeds keep their meaning. */
/* SimulateBeads.randomPoints (S/SimulateBeads.java:150-166), reference seed 535 (:69); host arithmetic; points = n x 3 (x, y, z) */
int mvsim_random_points(int n, const int64_t range_min[3], const int64_t range_max[3], int64_t seed, double* points);
/* SimulateBeads.transformPoints (:131-148) for one angle: axisRotation(range, axis, degrees) applied to every point; host arithmetic */
int mvsim_transform_points(const double* points, int n, const int64_t range_min[3], const int64_t range_max[3], int axis, int degrees, double* out);
/* SimulateBeads.renderPoints / addGaussian (:97-121, :168-205) for one point list.  As in the reference (:106) the image has
 * max - min voxels per axis (one less than the interval's dimension); out has prod(max - min) floats.  Sums in point order. */
int mvsim_render_beads(mvsim_ctx* ctx, const double* points, int n, const double sigma[3], const int64_t interval_min[3],
                       const int64_t interval_max[3], float* out);
/* drawSpheres (S/SimulateMultiViewDataset.java:436-522) into a zeroed volume of dims; reference seed 464232194 (:76), minValue 0,
 * maxValue 1, scale 2.  n_small (nullable) receives the number of small spheres. */
int mvsim_draw_spheres(mvsim_ctx* ctx, const int64_t dims[3], double min_value, double max_value, int scale, int half_pixel, int64_t seed,
                       float* out, int64_t* n_small);
/* downSample2x (:394-423): out has prod(dims/2 - 1) floats */
int mvsim_downsample2x(mvsim_ctx* ctx, const float* in, const int64_t dims[3], float* out);
/* simulate(halfPixelOffset, rnd) (:371-392): the size^3 ground truth (reference size 289), rendered at 2x and down-sampled on the device */
int mvsim_simulate_phantom(mvsim_ctx* ctx, int size, int half_pixel, int64_t seed, float* out, int64_t* n_small);
/* Tools.makeSquare (S/Tools.java:315-349): out is the cube of the largest dimension */
int mvsim_make_square(mvsim_ctx* ctx, const float* in, const int64_t dims[3], float* out);

/* ---- device-resident volumes (SNR sweeps a la S/SimulateTileStitching.java:131-189) ------- */
int mvsim_volume_create(mvsim_ctx* ctx, const int64_t dims[3], mvsim_volume** vol);
/* non-owning handle over device memory the caller allocated (16-byte aligned; e.g. a buffer an NCCL broadcast fills); freeing the
 * handle leaves the memory alone */
int mvsim_volume_wrap(mvsim_ctx* ctx, const int64_t dims[3], void* device_ptr, mvsim_volume** vol);
int mvsim_volume_free(mvsim_ctx* ctx, mvsim_volume* vol);
int mvsim_volume_dims(const mvsim_volume* vol, int64_t dims[3]);
void* mvsim_volume_device_ptr(mvsim_volume* vol);
int mvsim_volume_upload(mvsim_ctx* ctx, mvsim_volume* vol, const float* host);       /* async if pinned */
int mvsim_volume_download(mvsim_ctx* ctx, const mvsim_volume* vol, float* host);     /* async if pinned */

int mvsim_dev_rotate_axis(mvsim_ctx* ctx, const mvsim_volume* in, mvsim_volume* out, int axis, int degrees);
int mvsim_dev_attenuate(mvsim_ctx* ctx, const mvsim_volume* in, mvsim_volume* out, double delta, int strict_reference);
int mvsim_dev_psf_normalize(mvsim_ctx* ctx, mvsim_volume* psf, double* sum_out /* nullable: no sync */);
/* psf must already be normalised (mvsim_dev_psf_normalize); the spectrum is rebuilt per call like :257 */
int mvsim_dev_convolve(mvsim_ctx* ctx, const mvsim_volume* img, const mvsim_volume* psf, mvsim_volume* out);
int mvsim_dev_adjust(mvsim_ctx* ctx, mvsim_volume* img, float min_value, float target_avg, double* correction_out /* nullable: no sync */);
int mvsim_dev_extract_slices(mvsim_ctx* ctx, const mvsim_volume* in, int inc, float snr, uint64_t seed, uint64_t stream, mvsim_volume* out);
/* extractSlices (:195-231) of Views.zeroMin(Views.interval(in, min, max)) (S/SimulateTileStitching.java:152-153,174) without
 * materialising the view: min/max inclusive (x, y, z); out dims (max0-min0+1, max1-min1+1, (max2-min2)/inc+1).  Bit-identical to
 * mvsim_dev_extract_slices of the dense cut with the same seed / stream.  MVSIM_EINVAL for a null pointer, in == out, inc < 1,
 * an interval outside in (min < 0, max >= dims or min > max on any axis) or mismatched out dims; MVSIM_EUNSUPPORTED for a tile
 * plane (max0-min0+1)*(max1-min1+1) of 2^32 voxels or more. */
int mvsim_dev_extract_interval(mvsim_ctx* ctx, const mvsim_volume* in, const int64_t min[3], const int64_t max[3], int inc,
                               float snr, uint64_t seed, uint64_t stream, mvsim_volume* out);
/* gt: ground truth, psf: raw PSF (normalised in place), out: X*Y*((Z-1)/inc+1) */
int mvsim_dev_simulate_view(mvsim_ctx* ctx, const mvsim_view_params* p, const mvsim_volume* gt, mvsim_volume* psf, mvsim_volume* out);
/* the view loop (:567-613) on a ground truth that is already resident (uploaded once, generated on the device, or received from
 * another GPU over NVLink when views are sharded across ranks); PSFs and results are host buffers as in mvsim_simulate_views */
int mvsim_dev_simulate_views(mvsim_ctx* ctx, int n_views, const mvsim_view_params* params, const mvsim_volume* gt,
                             float* const* psfs, float* const* outs);
/* mvsim_simulate_dataset on a ground truth that is already resident */
int mvsim_dev_simulate_dataset(mvsim_ctx* ctx, int n_all, const mvsim_view_params* params, const int32_t* align_degrees, float osem,
                               int n_views, const int32_t* views, const mvsim_volume* gt, float* const* psfs,
                               const mvsim_dataset_outputs* outs, float* sum_weights);
/* rotateAroundAxis(makeIsotropic(acq, inc), 0, degrees) (:588, :591) gathered straight from the acquired planes, bit-identical to
 * the two stages; acq: X*Y*Za, out: X*Y*((Za-1)*inc+1) */
int mvsim_dev_align_view(mvsim_ctx* ctx, const mvsim_volume* acq, int inc, int degrees, mvsim_volume* out);
/* the normalised rotate-back weight images of a dataset of n_all views (:576, :592, :615-646) from the dims and angles alone (the
 * weight image depends on y only, so no volume is read): writes view views[j] into out[j]; sum_weights (nullable) = :648-663.
 * Bit-identical to mvsim_normalize_weights over mvsim_rotate_axis(mvsim_weight_image(dims), 0, align_degrees[k]) for all k. */
int mvsim_dev_aligned_weights(mvsim_ctx* ctx, const int64_t dims[3], int n_all, const int32_t* align_degrees, float osem,
                              int n_out, const int32_t* views, mvsim_volume* const* out, mvsim_volume* sum_weights);
/* the generators writing straight into a device-resident volume (the ground truth never visits the host) */
int mvsim_dev_render_beads(mvsim_ctx* ctx, const double* points, int n, const double sigma[3], const int64_t interval_min[3],
                           const int64_t interval_max[3], mvsim_volume* out);
int mvsim_dev_simulate_phantom(mvsim_ctx* ctx, int size, int half_pixel, int64_t seed, mvsim_volume* out, int64_t* n_small);

/* ---- slab-decomposed convolution of one large volume across ranks (SURVEY section 8e, BASELINE config 5) -------
 * convolve (:253-264) for a volume that is distributed by z slabs over `world` GPUs (one process each).
 * Rank r holds planes [r*Z/world, (r+1)*Z/world) of the image and of the result; x and y passes are local, the
 * fused z pass runs on kx tiles after an all-to-all transpose and a second all-to-all brings the slabs back.
 * The library does the passes; the CALLER runs the two exchanges (NCCL all_to_all_single with equal splits)
 * on the bound buffers between the calls -- their layout is already the send / receive layout:
 *     prepare;  for block in 0..y_blocks-1:  forward_y(block); [all_to_all send->recv]; middle_z;
 *                                            [all_to_all recv->send]; inverse_y(block);   finish
 * world == 1 skips the exchanges (recv buffer unused).  All pointers are DEVICE pointers; the PSF must already
 * be normalised (mvsim_dev_psf_normalize).  Needs Z % world == 0 and (kx tile count) % world == 0. */
typedef struct mvsim_slabconv mvsim_slabconv;
int mvsim_slabconv_create(mvsim_ctx* ctx, const int64_t dims[3], const int64_t kdims[3], int rank, int world, mvsim_slabconv** plan);
int mvsim_slabconv_destroy(mvsim_ctx* ctx, mvsim_slabconv* plan);
/* info = { z_local, z0, y_blocks, exchange buffer size in complex64 elements, nfft_x, nfft_y, nfft_z, tiles_own } */
int mvsim_slabconv_info(const mvsim_slabconv* plan, int64_t info[8]);
int mvsim_slabconv_bind(mvsim_slabconv* plan, void* send_buffer, void* recv_buffer);
int mvsim_slabconv_prepare(mvsim_ctx* ctx, mvsim_slabconv* plan, const float* d_psf, const float* d_img_slab);
int mvsim_slabconv_forward_y(mvsim_ctx* ctx, mvsim_slabconv* plan, int block);
int mvsim_slabconv_middle_z(mvsim_ctx* ctx, mvsim_slabconv* plan);
int mvsim_slabconv_inverse_y(mvsim_ctx* ctx, mvsim_slabconv* plan, int block);
int mvsim_slabconv_finish(mvsim_ctx* ctx, mvsim_slabconv* plan, float* d_out_slab);
/* Peer-to-peer mode (same node, NVLink): instead of bind + two all-to-alls per block, the library allocates nbuf (1 or 2)
 * buffer sets and exports 2*nbuf CUDA IPC handles of 64 bytes; after the ranks exchanged them (any transport), _p2p_open maps
 * the peers' buffers.  forward_y then stores each kx tile straight into the z-pass buffer of its owner and middle_z stores each
 * z slab straight into its owner's inverse-side buffer, so the transfers overlap the transforms tile by tile.  The caller only
 * places a cross-rank barrier (e.g. a 1-element all-reduce on the same stream) after forward_y and after middle_z:
 *     prepare;  for block: p2p_select(block % nbuf); forward_y(block); [barrier]; middle_z; [barrier]; inverse_y(block);  finish */
int mvsim_slabconv_p2p_alloc(mvsim_ctx* ctx, mvsim_slabconv* plan, int nbuf, unsigned char* handles_out /* 2*nbuf*64 bytes */);
int mvsim_slabconv_p2p_open(mvsim_ctx* ctx, mvsim_slabconv* plan, const unsigned char* all_handles /* world*2*nbuf*64 bytes, rank major */);
int mvsim_slabconv_p2p_select(mvsim_slabconv* plan, int buffer_set);


/* ---- the stages around the decomposed convolution: ONE view of a volume distributed by z slabs (DEVICE pointers) ----------
 * rank r owns the output planes [z0, z0 + z_local) of every stage.  Order, mirroring the loop body S/SimulateMultiViewDataset.java:570-585:
 *   mvsim_slab_rotate_attenuate (:570,573)  -> mvsim_slabconv_* (:580) -> mvsim_slab_sum, [all-gather of `world` doubles, rank order],
 *   mvsim_slab_adjust (:582, Tools.adjustImage S/Tools.java:143-159) -> mvsim_slab_extract (:585).
 * The ground truth stays WHOLE on every rank (generated there or broadcast over NVLink): a rotation about x reads source planes far
 * outside the output slab.  Only rotations about axis 0 (the reference's) are decomposed. */
int mvsim_slab_rotate_attenuate(mvsim_ctx* ctx, const float* d_gt, const int64_t dims[3], int axis, int degrees, double delta, int strict_reference,
                                int64_t z0, int64_t z_local, float* d_out_slab);
/* deterministic double sum of this rank's slab -> *d_sum (device memory) */
int mvsim_slab_sum(mvsim_ctx* ctx, const float* d_slab, size_t n_local, double* d_sum);
/* d_sums = the `world` per-rank sums in rank order (added in that order, so the correction is the same on every rank and does not depend on
 * the collective's reduction order); n_global = voxels of the whole volume.  In place: t = f32(f32(t * corr) + min_value). */
int mvsim_slab_adjust(mvsim_ctx* ctx, float* d_slab, size_t n_local, const double* d_sums, int world, double n_global, float min_value, float target_avg);
/* keeps the global planes z % inc == 0 that fall into the slab, compacted in order (*planes_out of them; d_out must hold
 * X*Y*((z_local-1)/inc+1) floats).  Philox counters are GLOBAL output voxel indices: the noise does not depend on the decomposition. */
int mvsim_slab_extract(mvsim_ctx* ctx, const float* d_slab, const int64_t dims[3], int64_t z0, int64_t z_local, int inc, float snr, uint64_t seed,
                       uint64_t stream, float* d_out, int64_t* planes_out);

#ifdef __cplusplus
}
#endif
#endif /* MVSIM_H */
