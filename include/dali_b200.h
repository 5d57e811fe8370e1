/*
 * include/dali_b200.h -- the thin C-ABI under the reference's operator boundary.
 *
 * Every hot-path kernel family is exposed as   plan create -> plan setup (host, per batch: shapes and
 * per-sample arguments) -> launch (enqueue on a caller stream, no host sync) -> plan destroy.
 * POD arguments only, caller owns every data buffer, the callee owns the plan and its pinned /
 * device descriptor arena.  Non-zero return = error; dalib200GetLastError() returns a thread-local
 * message (conventions follow the reference's C API: include/dali/dali.h:43-164).
 *
 * The reference has no such ABI (its kernels are C++ templates: Setup()/Run(ctx,out,in,args),
 * dali/kernels/kernel.h); each entry point below names the reference interface it replaces.
 * The C++ operators in dali_b200/host (Operator<GPUBackend>::SetupImpl / RunImpl, reference
 * dali/pipeline/operator/operator.h:117-123) call PlanSetup from SetupImpl and Launch from RunImpl.
 */
#ifndef DALI_B200_H_
#define DALI_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st *dalib200Stream_t;   /* == cudaStream_t */

/* Data type ids equal the reference's DALIDataType (include/dali/core/dali_data_type.h:44-57). */
enum { DALIB200_UINT8 = 0, DALIB200_INT16 = 5, DALIB200_FLOAT16 = 8, DALIB200_FLOAT = 9 };
/* Image types equal DALIImageType (include/dali/core/common.h:156-162). */
enum { DALIB200_RGB = 0, DALIB200_BGR = 1, DALIB200_GRAY = 2, DALIB200_YCbCr = 3 };
/* Resampling filters equal kernels::ResamplingFilterType (dali/kernels/imgproc/resample/params.h:27-34). */
enum { DALIB200_FILTER_NN = 0, DALIB200_FILTER_LINEAR = 1, DALIB200_FILTER_TRIANGULAR = 2,
       DALIB200_FILTER_GAUSSIAN = 3, DALIB200_FILTER_CUBIC = 4, DALIB200_FILTER_LANCZOS3 = 5 };
enum { DALIB200_LAYOUT_HWC = 0, DALIB200_LAYOUT_CHW = 1 };

enum {
  DALIB200_SUCCESS = 0,
  DALIB200_ERROR_INVALID_ARGUMENT = 1,
  DALIB200_ERROR_UNSUPPORTED = 2,
  DALIB200_ERROR_CUDA = 3,
  DALIB200_ERROR_BAD_DATA = 4,
  DALIB200_ERROR_INTERNAL = 5
};

const char *dalib200GetLastError(void);
int dalib200GetVersion(void);
/* number of kernels this library has launched from the calling process (bench.py's gpu_launches) */
uint64_t dalib200GetLaunchCount(void);
/* Per-launch device timing with CUDA events on the launching stream (off by default).  Collect synchronises,
 * returns the records in launch order and clears the log. */
int dalib200ProfilingEnable(int on);
int dalib200ProfilingCollect(char *names, int name_stride, float *ms, int max, int *count);

/* ------------------------------------------------------------------------------------------------
 * JPEG decode (Huffman + dequant + IDCT + chroma upsampling + YCbCr->RGB): baseline sequential (self-synchronising parallel entropy
 * decode) and progressive (SOF2: scans in dependency waves, one warp per scan; spectral selection + successive approximation).
 * Replaces: imgcodec::ImageDecoder<MixedBackend>::RunImplImpl -> nvimgcodecDecoderDecode
 *           (dali/operators/imgcodec/image_decoder.h:613-882) and ParseSample (:473-499).
 * Host work: marker/table parse only.  Device work: everything arithmetic. */
typedef struct dalib200JpegPlan dalib200JpegPlan;

typedef struct {
  int32_t width, height;        /* decoded image size */
  int32_t components;           /* 1 or 3 */
  int32_t subsampling;          /* (hmax<<4)|vmax of the luma sampling factors, e.g. 0x22 = 4:2:0 */
  int32_t restart_interval;
  int32_t orientation;          /* EXIF orientation, 1 = none */
} dalib200JpegInfo;

/* header-only parse: the analogue of nvimgcodecCodeStreamGetImageInfo (image_decoder.h:482) */
int dalib200JpegGetInfo(const uint8_t *data, size_t len, dalib200JpegInfo *info);

int dalib200JpegPlanCreate(dalib200JpegPlan **plan, int max_batch);
int dalib200JpegPlanDestroy(dalib200JpegPlan *plan);
/* Parses n encoded streams (host pointers) and builds the per-sample descriptors.  The streams are BORROWED until
 * dalib200JpegUpload returns (it packs the entropy-coded segments into the plan's pinned staging buffer, in groups, and
 * issues the H2D copy of each group as soon as it is packed).  Output shapes via ...GetInfo().
 * fancy_upsampling != 0 selects libjpeg "fancy" (triangle) chroma upsampling -- the reference CPU
 * backend's behaviour; 0 = box replication. */
int dalib200JpegPlanSetup(dalib200JpegPlan *plan, int n, const uint8_t *const *streams, const size_t *lengths,
                          int output_type /* DALIB200_RGB | BGR | GRAY */, int fancy_upsampling);
int dalib200JpegPlanGetInfo(const dalib200JpegPlan *plan, int sample, dalib200JpegInfo *info);
/* Full argument surface of the decoder operators (decoders.image / image_crop / image_random_crop / image_slice):
 *   output_type          DALIB200_RGB | BGR | GRAY | YCbCr   (decoder_schema.cc:21-60; YCbCr = BT.601 of the decoded RGB,
 *                        dali/operators/imgcodec/util/convert.h:150-160)
 *   dtype                DALIB200_UINT8 | DALIB200_FLOAT     (ConvertSatNorm: u8 * (1 / 255), convert.h:118-128)
 *   adjust_orientation   apply the EXIF orientation (image_decoder.h:211,678-679,806)
 *   rois[i]              region of interest of sample i in OUTPUT (oriented) pixel coordinates, [x0, x1) x [y0, y1)
 *                        (imgcodec.h:26-44, image_decoder.h:681-716); only the MCUs under the region are transformed.
 * The result equals the full decode followed by orientation, crop and conversion, bit for bit. */
typedef struct { int32_t output_type, fancy_upsampling, dtype, adjust_orientation; } dalib200JpegParams;
typedef struct {
  int32_t use_roi, x0, y0, x1, y1;
  int32_t planes_only;        /* skip upsampling + colour conversion for this sample: the caller reads the component planes
                                 (dalib200JpegPlanGetPlanes -> dalib200ResampleLaunchPlanar); 4:2:0 YCbCr streams only */
} dalib200JpegRoi;
/* The decoder's planar output of a sample: 8-bit planes, Cb / Cr at half resolution (4:2:0), rows padded to a multiple of 16 bytes.
 * Only the MCUs under the sample's region of interest hold data.  crop_x / crop_y: filled by the caller (window the resampler treats
 * as its input image). */
typedef struct {
  const uint8_t *y, *cb, *cr;
  int32_t pitch_y, pitch_c;
  int32_t width, height;
  int32_t crop_x, crop_y;
} dalib200PlanarImage;
/* Alternative to the planes_only flags of SetupEx, for callers that learn only after the setup which samples they can consume as
 * planes: want[i] != 0 asks for sample i, granted[i] tells whether the stream qualifies (3 components, 4:2:0, YCbCr, fancy upsampling,
 * no orientation, RGB u8 request).  Call between JpegPlanSetupEx and JpegUpload. */
int dalib200JpegPlanSetPlanesOnly(dalib200JpegPlan *plan, const uint8_t *want, uint8_t *granted);
/* valid after dalib200JpegLaunch of the batch (the plane arena may grow there) until the next launch */
int dalib200JpegPlanGetPlanes(const dalib200JpegPlan *plan, int sample, dalib200PlanarImage *out);
int dalib200JpegPlanSetupEx(dalib200JpegPlan *plan, int n, const uint8_t *const *streams, const size_t *lengths,
                            const dalib200JpegParams *params, const dalib200JpegRoi *rois_or_null);
/* (H, W, C) of the sample the launch will write (after orientation and region of interest) */
int dalib200JpegPlanGetOutputShape(const dalib200JpegPlan *plan, int sample, int32_t *hwc);
/* Bytes of packed entropy-coded data + tables staged for the batch (the H2D payload). */
size_t dalib200JpegPlanStagedBytes(const dalib200JpegPlan *plan);
/* Pinned staging + H2D copy of the batch (async on stream, host work overlapped with the transfer).  Split from Launch
 * so that a caller can time the device-resident decode separately from the transfer. */
int dalib200JpegUpload(dalib200JpegPlan *plan, dalib200Stream_t stream);
/* stable != 0: the caller guarantees that the encoded streams passed to the next JpegPlanSetup calls stay valid and unmodified
 * until the launch that consumes them has completed -- the contract of the reference's external_source(no_copy=True)
 * (dali/python/nvidia/dali/external_source.py, `no_copy`) and of its readers' own buffers.  JpegUpload then copies samples that
 * live in page-locked memory straight from the caller's buffers (one DMA per sample, no host repack); anything else still goes
 * through the pinned staging buffer.  JpegPlanLastUploadDirect: 0 = staged, 1 = direct (one cudaMemcpyAsync per
 * sample), 2 = direct as one cudaMemcpyBatchAsync submission. */
int dalib200JpegPlanSetSourceStable(dalib200JpegPlan *plan, int stable);
int dalib200JpegPlanLastUploadDirect(const dalib200JpegPlan *plan);
/* Test hook: exhaustive (2^32 inputs) check of the kernels' float -> float16 conversion against the integer restatement of the
 * reference's half_float rounding (include/dali/util/half.hpp, ties away from zero).  *mismatches == 0 on success. */
int dalib200DebugCheckHalfConversion(uint64_t *mismatches);
/* Page-locked host memory for callers that want the direct path (cudaHostAlloc / cudaFreeHost behind the C ABI). */
int dalib200HostAlloc(void **ptr, size_t bytes);
/* The same from a thread whose current device is not the consumer's: allocated with `device` current (no context appears on another
 * GPU as a side effect), page-locked for every context (cudaHostAllocPortable); the thread's current device is restored. */
int dalib200HostAllocOnDevice(void **ptr, size_t bytes, int device);
int dalib200HostFree(void *ptr);
/* Enqueues the decode of the uploaded batch; out_ptrs[i] -> device buffer H*W*C of dtype (HWC, see ...GetOutputShape). */
int dalib200JpegLaunch(dalib200JpegPlan *plan, void *const *out_ptrs, dalib200Stream_t stream);
/* Per-sample device status after a launch (0 ok, 1 = entropy-coded data ended early).  Synchronises. */
int dalib200JpegGetStatus(dalib200JpegPlan *plan, int32_t *status_out);
/* Non-blocking status: ...Async enqueues the D2H copy of the status words on `stream` into the plan's pinned buffer, ...Fetch reads
 * them once the caller has synchronised the stream (the operator does it where the executor waits for the outputs, so a truncated
 * stream raises from Pipeline.run() without an extra synchronisation). */
int dalib200JpegStatusAsync(dalib200JpegPlan *plan, dalib200Stream_t stream);
int dalib200JpegStatusFetch(const dalib200JpegPlan *plan, int32_t *status_out, int n);
/* Test accessor: quantised coefficients of one sample (MCU order, natural order per block).  Synchronises. */
int dalib200JpegDebugGetCoefficients(dalib200JpegPlan *plan, int sample, int16_t *out, size_t count);

/* ------------------------------------------------------------------------------------------------
 * Separable resampling (fused two-pass).  Replaces kernels::ResampleGPU / SeparableResamplingGPUImpl::Run
 * (dali/kernels/imgproc/resample/separable_impl.h:110-203) and BatchResamplingSetup::SetupBatch
 * (resampling_setup.cc:347-418); numerics follow the CPU kernel SeparableResampleCPU
 * (separable_cpu.h:124-249) -- the parity target. */
typedef struct dalib200ResamplePlan dalib200ResamplePlan;

typedef struct { int32_t type; int32_t antialias; float radius; } dalib200FilterDesc;

typedef struct {
  int32_t in_h, in_w, channels;
  int32_t out_h, out_w;
  /* index [0] = vertical (y), [1] = horizontal (x): the reference's ResamplingParams2D order */
  int32_t use_roi[2];
  float roi_start[2], roi_end[2];
  dalib200FilterDesc min_filter[2], mag_filter[2];
} dalib200ResampleSample;

int dalib200ResamplePlanCreate(dalib200ResamplePlan **plan, int max_batch);
int dalib200ResamplePlanDestroy(dalib200ResamplePlan *plan);
int dalib200ResamplePlanSetup(dalib200ResamplePlan *plan, int n, const dalib200ResampleSample *samples,
                              int in_dtype /* UINT8 | FLOAT */, int out_dtype /* UINT8 | FLOAT */);
/* in_ptrs[i]: device HWC in_dtype; out_ptrs[i]: device HWC out_dtype [out_h][out_w][channels] */
int dalib200ResampleLaunch(dalib200ResamplePlan *plan, const void *const *in_ptrs, void *const *out_ptrs,
                           dalib200Stream_t stream);
/* Decode -> resize without the RGB image (SURVEY.md 8f rank 1: the reference's fused ROI decode + resize path,
 * image_decoder.h:699-716 + resize.cc): samples whose `planar_ok` is 1 after ...SetupPlanar are resampled straight from the decoder's
 * planes (fancy chroma upsampling + YCbCr->RGB happen inside the resampling kernel, bit-exact with decode-then-resize); sample i of
 * ...LaunchPlanar reads srcs[i] (window crop_x, crop_y, in_w x in_h of the setup) and is skipped when planar_ok[i] == 0. */
int dalib200ResamplePlanSetupPlanar(dalib200ResamplePlan *plan, int n, const dalib200ResampleSample *samples, uint8_t *planar_ok);
int dalib200ResampleLaunchPlanar(dalib200ResamplePlan *plan, const dalib200PlanarImage *srcs, void *const *out_ptrs,
                                 dalib200Stream_t stream);
/* introspection used by the tests: processing order chosen for a sample (0 = horizontal pass first) */
int dalib200ResamplePlanGetOrder(const dalib200ResamplePlan *plan, int sample);
/* 1 when the sample went through the streaming (TMA ring) kernel in the last launch, 0 = tile kernel, -1 = bad index. */
int dalib200ResamplePlanGetPath(const dalib200ResamplePlan *plan, int sample);

/* ------------------------------------------------------------------------------------------------
 * Separable resampling of volumes (DHWC), three passes.  Replaces the spatial_ndim = 3 instances of kernels::ResampleGPU /
 * SeparableResamplingGPUImpl (dali/kernels/imgproc/resample/separable_impl.h:110-203, resampling_setup.cc:232-337) behind
 * ResizeBase<GPUBackend> (dali/operators/image/resize/resize_base.cc, resize_op_impl_gpu.h); numerics follow
 * SeparableResampleCPU<Out, In, 3> (separable_cpu.h:124-249) -- the parity target. */
typedef struct dalib200Resample3DPlan dalib200Resample3DPlan;

typedef struct {
  /* index [0] = depth (z), [1] = height (y), [2] = width (x): shape order = the reference's ResamplingParams3D order */
  int32_t in_shape[3], channels;
  int32_t out_shape[3];
  int32_t use_roi[3];
  float roi_start[3], roi_end[3];
  dalib200FilterDesc min_filter[3], mag_filter[3];
} dalib200Resample3DSample;

int dalib200Resample3DPlanCreate(dalib200Resample3DPlan **plan, int max_batch);
int dalib200Resample3DPlanDestroy(dalib200Resample3DPlan *plan);
int dalib200Resample3DPlanSetup(dalib200Resample3DPlan *plan, int n, const dalib200Resample3DSample *samples,
                                int in_dtype /* UINT8 | FLOAT */, int out_dtype /* UINT8 | FLOAT */);
/* in_ptrs[i]: device DHWC in_dtype; out_ptrs[i]: device DHWC out_dtype [out_shape][channels] */
int dalib200Resample3DLaunch(dalib200Resample3DPlan *plan, const void *const *in_ptrs, void *const *out_ptrs, dalib200Stream_t stream);
/* introspection used by the tests: the pass order chosen for a sample, axes numbered 0 = x (width), 1 = y, 2 = z (depth) */
int dalib200Resample3DPlanGetOrder(const dalib200Resample3DPlan *plan, int sample, int32_t order[3]);

/* ------------------------------------------------------------------------------------------------
 * CropMirrorNormalize.  Replaces kernels::SliceHwc2HwcChwNormalizeGPU::Run
 * (dali/kernels/slice/slice_hwc2chw_normalize_gpu.cu:863-1020) and the generic SliceFlipNormalize kernels;
 * numerics follow SliceFlipNormalizePermutePadCpu (slice_flip_normalize_permute_pad_cpu.h:37-46). */
typedef struct dalib200CmnPlan dalib200CmnPlan;

typedef struct {
  int32_t in_h, in_w, channels;              /* u8 HWC input */
  int32_t anchor_y, anchor_x, crop_h, crop_w;/* window in input coordinates; may leave the image (padding) */
  int32_t mirror;                            /* flip the cropped window horizontally */
  float mean[4], inv_std[4], fill[4];        /* per OUTPUT channel */
} dalib200CmnSample;

int dalib200CmnPlanCreate(dalib200CmnPlan **plan, int max_batch);
int dalib200CmnPlanDestroy(dalib200CmnPlan *plan);
int dalib200CmnPlanSetup(dalib200CmnPlan *plan, int n, const dalib200CmnSample *samples,
                         int out_dtype /* FLOAT | FLOAT16 */, int out_layout /* HWC | CHW */, int out_channels);
int dalib200CmnLaunch(dalib200CmnPlan *plan, const void *const *in_ptrs, void *const *out_ptrs, dalib200Stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * WarpAffine.  Replaces kernels::WarpGPU<AffineMapping2D,...> (dali/kernels/imgproc/warp_gpu.h,
 * warp/warp_variable_size_impl.cuh:31-42); numerics follow WarpCPU (warp_cpu.h:143-178) and
 * Sampler (sampler.h:122-330). */
typedef struct dalib200WarpPlan dalib200WarpPlan;

typedef struct {
  int32_t in_h, in_w, channels;
  int32_t out_h, out_w;
  float matrix[6];            /* 2x3 row-major DESTINATION -> SOURCE map (already inverted if needed) */
} dalib200WarpSample;

int dalib200WarpPlanCreate(dalib200WarpPlan **plan, int max_batch);
int dalib200WarpPlanDestroy(dalib200WarpPlan *plan);
int dalib200WarpPlanSetup(dalib200WarpPlan *plan, int n, const dalib200WarpSample *samples,
                          int interp /* NN | LINEAR */, int use_fill, float fill_value,
                          int out_dtype /* UINT8 | FLOAT */);
int dalib200WarpLaunch(dalib200WarpPlan *plan, const void *const *in_ptrs, void *const *out_ptrs, dalib200Stream_t stream);
/* Kernel taken by the last launch: 1 = band kernel with the source boxes staged by tiled TMA loads through a tensor map (bilinear
 * u8 -> u8 over 3-channel frames of one shape laid out at a constant 16-byte-aligned stride, e.g. the frames of an FHWC batch);
 * 2 = band kernel without a tensor map (bilinear u8 -> u8, 3 channels, any shapes); 0 = generic kernel (NN, float output, other
 * channel counts). */
int dalib200WarpPlanGetPath(const dalib200WarpPlan *plan);
/* host helper: include/dali/core/geom/transform.h:166-174 */
void dalib200AffineInverse(const float *m2x3, float *out2x3);

/* ------------------------------------------------------------------------------------------------
 * Per-pixel 3x3 linear colour transform (Hsv / ColorTwist) and colour-space conversion.
 * Replaces kernels::LinearTransformationGpu (pointwise/linear_transformation_gpu.h:47-79) and
 * ColorSpaceConvKernel (color_manipulation/color_space_conversion_kernel.cuh:139-211). */
typedef struct dalib200PointwisePlan dalib200PointwisePlan;

typedef struct {
  int64_t num_pixels;
  float matrix[9];          /* row-major 3x3 */
  float offset[3];
} dalib200ColorSample;

int dalib200PointwisePlanCreate(dalib200PointwisePlan **plan, int max_batch);
int dalib200PointwisePlanDestroy(dalib200PointwisePlan *plan);
int dalib200LinearTransformSetup(dalib200PointwisePlan *plan, int n, const dalib200ColorSample *samples,
                                 int out_dtype /* UINT8 | FLOAT */);
int dalib200ColorSpaceSetup(dalib200PointwisePlan *plan, int n, const int64_t *num_pixels, int in_type, int out_type);
int dalib200PointwiseLaunch(dalib200PointwisePlan *plan, const void *const *in_ptrs, void *const *out_ptrs,
                            dalib200Stream_t stream);
/* host helper: dali/operators/image/color/color_twist.h:50-83,156-170 */
void dalib200ColorTwistMatrix(float hue, float saturation, float value, float brightness, float contrast,
                              float half_range, float *m3x3, float *offset3);

/* ------------------------------------------------------------------------------------------------
 * Spectrogram (window extraction + FFT + |X|^p) and MelFilterBank.
 * Replaces kernels::signal::fft::StftGPU (dali/kernels/signal/fft/stft_gpu_impl.cu:200-294, cuFFT) and
 * kernels::audio::MelFilterBankGpu (audio/mel_scale/mel_filter_bank_gpu.cu:76-261). */
typedef struct dalib200SpectrogramPlan dalib200SpectrogramPlan;

typedef struct {
  int32_t nfft, window_length, window_step;
  int32_t power;             /* 1 = magnitude, 2 = power */
  int32_t center, reflect;   /* center_windows / reflect_padding */
  int32_t layout_ft;         /* 1: [freq][time] (default "ft"), 0: [time][freq] */
} dalib200SpectrogramArgs;

int dalib200SpectrogramPlanCreate(dalib200SpectrogramPlan **plan, int max_batch);
int dalib200SpectrogramPlanDestroy(dalib200SpectrogramPlan *plan);
/* window_fn: host pointer to window_length floats, or NULL for the reference's Hann window */
int dalib200SpectrogramPlanSetup(dalib200SpectrogramPlan *plan, const dalib200SpectrogramArgs *args,
                                 const float *window_fn, int n, const int64_t *lengths);
int64_t dalib200SpectrogramNumWindows(const dalib200SpectrogramPlan *plan, int sample);
int dalib200SpectrogramLaunch(dalib200SpectrogramPlan *plan, const void *const *in_ptrs, void *const *out_ptrs,
                              dalib200Stream_t stream);
void dalib200HannWindow(float *out, int n);

typedef struct dalib200MelPlan dalib200MelPlan;

typedef struct {
  int32_t nfilter;
  float sample_rate, freq_low, freq_high;
  int32_t htk;               /* mel_formula == "htk" */
  int32_t normalize;
} dalib200MelArgs;

int dalib200MelPlanCreate(dalib200MelPlan **plan, int max_batch);
int dalib200MelPlanDestroy(dalib200MelPlan *plan);
/* input spectrograms are [nbin][nwin[i]] f32 ("ft"); outputs [nfilter][nwin[i]] */
int dalib200MelPlanSetup(dalib200MelPlan *plan, const dalib200MelArgs *args, int nbin, int n, const int64_t *nwin);
/* enable != 0: run the filter bank as one dense GEMM on the tensor cores (mma.sync TF32, 3-term split, FP32 accumulate).
 * Tolerance path (summation order differs from the reference CPU kernel, ~1e-6 relative); the default (0) is the bit-exact
 * banded kernel. */
int dalib200MelPlanSetTensorCores(dalib200MelPlan *plan, int enable);
int dalib200MelLaunch(dalib200MelPlan *plan, const void *const *in_ptrs, void *const *out_ptrs, dalib200Stream_t stream);
/* Spectrogram -> MelFilterBank in ONE kernel (audio/mel_scale/mel_filter_bank.cc consuming signal/fft/spectrogram.cc): the
 * power spectrum of a frame pair stays in shared memory and only the nfilter x nwin mel output is written.  Available for
 * nfft = 1024 with the (f, t) layout and a mel plan set up for the same batch (dalib200SpectrogramMelSupported returns 1).
 * spec_out_ptrs may be NULL: the spectrogram is then not materialised at all. */
int dalib200SpectrogramMelSupported(const dalib200SpectrogramPlan *plan, const dalib200MelPlan *mel);
int dalib200SpectrogramMelLaunch(dalib200SpectrogramPlan *plan, dalib200MelPlan *mel, const void *const *in_ptrs,
                                 void *const *spec_out_ptrs, void *const *mel_out_ptrs, dalib200Stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Audio tail behind Spectrogram / MelFilterBank: ToDecibels, MFCC (DCT + liftering), Normalize.
 * Replaces kernels::signal::ToDecibelsGpu (dali/kernels/signal/decibel/to_decibels_gpu.cu), kernels::signal::dct::Dct1DGpu
 * (dali/kernels/signal/dct/dct_gpu.cu) + the liftering of dali/operators/audio/mfcc/mfcc.cu, and the 2-D float case of
 * kernels::NormalizeGPU (dali/kernels/normalize/normalize_gpu.cu); numerics follow the CPU kernels
 * (to_decibels_cpu.cc:47-72, dct_cpu.cc:76-115, mfcc.cc:52-72). */
typedef struct dalib200SignalPlan dalib200SignalPlan;
typedef struct {
  float multiplier, reference, cutoff_db;   /* dali/operators/signal/decibel/to_decibels_op.h:38-50 */
  int32_t ref_max;                          /* no `reference` given: the per-sample maximum is the reference */
} dalib200ToDecibelsArgs;
typedef struct { int32_t n_mfcc, dct_type, normalize; float lifter; } dalib200MfccArgs;
typedef struct {
  int32_t mode;                             /* 0: reduce both axes, 1: reduce axis 1 (per row), 2: reduce axis 0 (per column) */
  int32_t ddof;
  float scale, shift, epsilon;
} dalib200NormalizeArgs;

int dalib200SignalPlanCreate(dalib200SignalPlan **plan, int max_batch);
int dalib200SignalPlanDestroy(dalib200SignalPlan *plan);
int dalib200ToDecibelsSetup(dalib200SignalPlan *plan, const dalib200ToDecibelsArgs *args, int n, const int64_t *volumes);
/* shapes: n x 2 = (features, frames); the transform runs along axis 0; outputs are [min(n_mfcc, features)][frames] */
int dalib200MfccSetup(dalib200SignalPlan *plan, const dalib200MfccArgs *args, int n, const int64_t *shapes);
int dalib200SignalOutputRows(const dalib200SignalPlan *plan);
int dalib200NormalizeSetup(dalib200SignalPlan *plan, const dalib200NormalizeArgs *args, int n, const int64_t *shapes);
/* in_ptrs[i] / out_ptrs[i]: device f32 */
int dalib200SignalLaunch(dalib200SignalPlan *plan, const void *const *in_ptrs, void *const *out_ptrs, dalib200Stream_t stream);

/* AudioResample (dali/operators/audio/resample.{h,cc}, kernel dali/kernels/signal/resampling_cpu.cc): float in, float out, 1..8
 * interleaved channels; in_rate / out_rate as the operator derives them (scale: 1 / scale; out_length: in_length / out_length);
 * out_length = resampled_length() = ceil(in_length * out_rate / in_rate) unless given.  quality 0..100 selects the windowed-sinc
 * width (resampling_params.h).  Launched with dalib200SignalLaunch. */
typedef struct {
  double in_rate, out_rate;
  int64_t in_length, out_length;
  int32_t channels;
} dalib200AudioResampleSample;
int dalib200AudioResampleSetup(dalib200SignalPlan *plan, int n, const dalib200AudioResampleSample *samples, float quality);

/* NonsilentRegion (dali/operators/audio/nonsilence_op.{h,cc}; moving mean square: dali/kernels/signal/moving_mean_square.cc):
 * float input, two int32 scalars per sample (begin, length).  use_reference_power == 0: the reference is the maximum of the
 * moving mean square (the operator's default).  reset_interval: -1 or a multiple of window_length (float inputs: 8192). */
typedef struct {
  float cutoff_db;
  float reference_power;
  int32_t use_reference_power;
} dalib200NonsilentSample;
int dalib200NonsilentSetup(dalib200SignalPlan *plan, int n, const int64_t *lengths, const dalib200NonsilentSample *args,
                           int window_length, int reset_interval);
int dalib200NonsilentLaunch(dalib200SignalPlan *plan, const void *const *in_ptrs, void *const *begin_ptrs,
                            void *const *length_ptrs, dalib200Stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Small per-pixel / geometry helpers (SURVEY.md 8f rank 4) for interleaved u8 images:
 *   multiply-add   out = ConvertSat<Out>(in * multiplier + addend)   -- brightness_contrast
 *                  (kernels::MultiplyAddGpu, dali/kernels/imgproc/pointwise/multiply_add_gpu.h; CPU numerics multiply_add.h:47-60)
 *   window copy    crop / slice / flip with out-of-bounds fill        -- fn.crop, fn.slice, fn.flip
 *                  (kernels::SliceGPU / SliceFlipNormalizePermutePadGpu, dali/kernels/slice/) */
typedef struct dalib200GenericPlan dalib200GenericPlan;
typedef struct {
  int32_t in_h, in_w, channels;
  int32_t anchor_y, anchor_x, out_h, out_w;   /* window in input coordinates; may leave the image (filled) */
  int32_t flip_x, flip_y;                     /* mirror the window horizontally / vertically */
  uint8_t fill[4];                            /* per channel */
} dalib200WindowSample;
int dalib200GenericPlanCreate(dalib200GenericPlan **plan, int max_batch);
int dalib200GenericPlanDestroy(dalib200GenericPlan *plan);
int dalib200MultiplyAddSetup(dalib200GenericPlan *plan, int n, const int64_t *volumes, const float *multipliers,
                             const float *addends, int out_dtype /* UINT8 | FLOAT */);
int dalib200WindowCopySetup(dalib200GenericPlan *plan, int n, const dalib200WindowSample *samples);
int dalib200GenericLaunch(dalib200GenericPlan *plan, const void *const *in_ptrs, void *const *out_ptrs, dalib200Stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Separable convolution with reflect-101 borders (fn.gaussian_blur).  Replaces kernels::SeparableConvolutionGpu
 * (dali/kernels/imgproc/convolution/separable_convolution_gpu.h) behind GaussianBlurOpGpu
 * (dali/operators/image/convolution/gaussian_blur_gpu.cu); numerics follow SeparableConvolutionCpu
 * (separable_convolution_cpu.h, convolution_cpu.h) -- the parity target: passes innermost axis first, fp32 intermediates,
 * taps summed in ascending order with separately rounded products and sums.
 * A sample is one channel-last 2-D frame (HW / HWC) or volume (DHW / DHWC); the caller flattens sequences into frames. */
typedef struct dalib200SepConvPlan dalib200SepConvPlan;

typedef struct {
  int32_t ndim;               /* spatial rank: 2 or 3 */
  int32_t shape[3];           /* spatial extents, outermost first: (H, W) or (D, H, W) */
  int32_t channels;
  int32_t diameter[3];        /* window length per axis, same order; odd, 1 .. 8191 */
  int32_t window_offset[3];   /* first tap of each axis' window in the caller's window array */
} dalib200SepConvSample;

int dalib200SepConvPlanCreate(dalib200SepConvPlan **plan, int max_batch);
int dalib200SepConvPlanDestroy(dalib200SepConvPlan *plan);
/* windows: host array of num_window_floats taps that the samples index into (windows shared by several samples are stored once
 * in the plan's coefficient table).  in_dtype / out_dtype: u8 -> u8, u8 -> f32, f32 -> f32. */
int dalib200SepConvPlanSetup(dalib200SepConvPlan *plan, int n, const dalib200SepConvSample *samples, const float *windows,
                             int64_t num_window_floats, int in_dtype, int out_dtype);
/* in_ptrs[i] / out_ptrs[i]: device buffers of the sample's shape x channels (output shape = input shape) */
int dalib200SepConvLaunch(dalib200SepConvPlan *plan, const void *const *in_ptrs, void *const *out_ptrs, dalib200Stream_t stream);
/* introspection used by the tests: 1 = streaming 2-D kernel (TMA row ring), 0 = per-axis pass kernels, -1 = bad index.  The path of
 * the last launch (before the first launch: the setup's choice, which a launch demotes to 0 for an input not 16-byte aligned). */
int dalib200SepConvPlanGetPath(const dalib200SepConvPlan *plan, int sample);
/* host helper: FillGaussian (dali/operators/image/convolution/gaussian_blur_params.h) -- `diameter` taps of the normalised Gaussian
 * of `sigma`, computed in double and rounded to float per tap */
void dalib200GaussianWindow(float sigma, int diameter, float *out);

#ifdef __cplusplus
}
#endif
#endif  /* DALI_B200_H_ */
