/* b200iop.h -- C ABI of libb200iop.so: the Ansel develop-pixelpipe hot path on B200 (sm_100a).
 *
 * Drop-in boundary (SURVEY.md section 8b).  A reference module keeps its dt_iop_module_t
 * surface (src/iop/iop_api.h:80-351) in plain C and forwards the body of
 *     process()            iop_api.h:265-266   -> b200_<op>_process_host()   host pointers, H2D + kernels + D2H
 *     process_cl()         iop_api.h:292-293   -> b200_<op>_process_dev()    device pointers + stream, no copies
 *     tiling_callback()    iop_api.h:121-122   -> b200_<op>_tiling()
 * to this library.  ansel_b200/iop/ holds those C adapters; INTEGRATION.md shows where they slot
 * into the reference tree.  No C++/CUDA/torch type crosses this header: plain pointers, sizes,
 * and PODs whose layout mirrors the reference structs they stand for (each cited below).
 *
 * Return convention of every int-returning entry point: 0 = success, non-zero = error
 * (b200_last_error() describes it).  That is process()'s convention (develop/pixelpipe_cpu.c:117-133);
 * a process_cl() adapter returns `rc == 0` because that slot means TRUE = success
 * (develop/pixelpipe_gpu.c:358).
 *
 * Threading: entry points are re-entrant.  Any number of threads may run the same module at once, each on its own
 * stream(s), as the reference's pipes do (doc/reorganisation.md:77-81): the darkroom's preview and full pipes, the frames
 * of a batch export.  Device scratch and the geometry plans of the demosaicers are per calling thread and per device.
 * One thread that drives several streams must order the modules that share its scratch, as b200_pixelpipe_submit does
 * with its `compute_done` events.
 * There is no CPU fallback anywhere in this library: without a CUDA device calls fail.
 */
#ifndef B200IOP_H
#define B200IOP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_ABI_VERSION 1

/* ---- error codes ------------------------------------------------------------------------ */
enum
{
  B200_OK = 0,
  B200_ERR_CUDA = 1,        /* a CUDA runtime/driver call failed */
  B200_ERR_ARG = 2,         /* NULL / inconsistent arguments */
  B200_ERR_UNSUPPORTED = 3, /* valid in the reference, not built here (say so, never guess) */
  B200_ERR_NODEVICE = 4,    /* no usable sm_100 device */
  B200_ERR_NOMEM = 5
};

/* ---- mirrors of the reference's operator-surface types ----------------------------------- */

/* dt_iop_roi_t, src/pixel/format.h:48-52 (identical layout) */
typedef struct b200_roi_t
{
  int x, y, width, height;
  double scale;
} b200_roi_t;

/* dt_develop_tiling_t, src/develop/tiling.h:39-58 (identical layout) */
typedef struct b200_tiling_t
{
  float factor, factor_cl, maxbuf, maxbuf_cl;
  unsigned overhead, overlap, xalign, yalign;
} b200_tiling_t;

/* dt_dev_pixelpipe_type_t, src/develop/pixelpipe.h:41-45 (same values) */
enum
{
  B200_PIPE_NONE = 0,
  B200_PIPE_EXPORT = 1,
  B200_PIPE_FULL = 2,
  B200_PIPE_PREVIEW = 3,
  B200_PIPE_THUMBNAIL = 4
};

/* dt_iop_buffer_type_t, src/pixel/format.h:54-59 (same values) */
enum
{
  B200_TYPE_UNKNOWN = 0,
  B200_TYPE_FLOAT = 1,
  B200_TYPE_UINT16 = 2,
  B200_TYPE_UINT8 = 3
};

/* Exactly the fields the hot-path process() bodies read from `piece`, `pipe` and `self`
 * (SURVEY.md appendix D): dt_dev_pixelpipe_iop_t src/develop/pixelpipe_hb.h:101-166,
 * dt_iop_buffer_dsc_t src/pixel/format.h:80-119. */
typedef struct b200_piece_t
{
  b200_roi_t roi_in, roi_out;  /* piece->roi_in / roi_out */
  uint32_t filters;            /* piece->dsc_in.filters (sensor phase only; the ROI shift of
                                  develop/imageop.c:139-142 is applied inside the library) */
  uint8_t xtrans[6][6];        /* piece->dsc_in.xtrans */
  uint32_t channels;           /* piece->dsc_in.channels */
  float processed_maximum[4];  /* piece->dsc_in.processed_maximum */
  float wb_coeffs[4];          /* piece->dsc_in.temperature.coeffs */
  int buf_in_width, buf_in_height; /* piece->buf_in */
  int pipe_type;               /* pipe->type */
  int mask_display;            /* pipe->mask_display */
  double iscale;               /* pipe->iscale */
  float exif_iso;              /* self->dev->image_storage.exif_iso */
  uint32_t image_flags;        /* self->dev->image_storage.flags */
  int devid;                   /* pipe->devid: CUDA device ordinal, < 0 = current device */
  int datatype;                /* piece->dsc_in.datatype (B200_TYPE_*); read by rawprepare only.  Occupies what was
                                  padding: the struct's size and every other offset are unchanged */
  const void *data;            /* piece->data: the module's b200_<op>_data_t */
  size_t data_size;            /* piece->data_size */
} b200_piece_t;

/* ---- library lifetime -------------------------------------------------------------------- */
int b200_abi_version(void);
/* Bind up to ndev devices (0 = all visible).  Fails with B200_ERR_NODEVICE when there is no
 * CUDA device -- there is no CPU path behind this ABI.  Stands where dt_opencl_init() does
 * (src/common/opencl.c). */
int b200_init(int ndev);
void b200_shutdown(void);
int b200_device_count(void);
/* thread-local, never NULL */
const char *b200_last_error(void);
/* Launch timing of the two headline kernels, for benchmarks: while enabled, every launch of `nlm_kernel` (whichever
 * non-local-means kernel the launcher picked: nlm.cu, nlm_group.cuh) and `rcd_tiles_kernel` (RCD demosaic, rcd.cu) is
 * bracketed by its own pair of CUDA events on the stream it is launched on, from any thread.
 * b200_kernel_timing(1) clears what was recorded and starts, (0) clears and stops;
 * b200_kernel_timing_read() waits for the recorded launches of one kernel and returns their summed duration and count.
 * No counterpart in the reference (its OpenCL path profiles through dt_opencl_events_*, src/common/opencl.c). */
int b200_kernel_timing(int enable);
int b200_kernel_timing_read(const char *kernel, double *sum_ms, int *count);

/* ---- device memory for callers that keep buffers resident between modules --------------------
 * The counterparts of dt_opencl_alloc_device_buffer / dt_opencl_copy_host_to_device /
 * dt_opencl_copy_device_to_host (src/common/opencl.c) used by pixelpipe_gpu.c:317-328,456-463.
 * `stream` is a cudaStream_t (NULL = default).  Pinned host memory is copied asynchronously;
 * pageable memory is staged. */
int b200_dev_alloc(void **ptr, size_t bytes);
void b200_dev_free(void *ptr);
int b200_copy_host_to_device(void *d_dst, const void *h_src, size_t bytes, void *stream);
int b200_copy_device_to_host(void *h_dst, const void *d_src, size_t bytes, void *stream);
int b200_stream_synchronize(void *stream);
/* streams and events for callers that keep several frames in flight (the reference's per-device command queues
 * and dt_opencl_events_*, src/common/opencl.c): non-blocking streams; events without timing */
int b200_stream_create(void **stream);
void b200_stream_destroy(void *stream);
int b200_event_create(void **event);
void b200_event_destroy(void *event);
int b200_event_record(void *event, void *stream);
int b200_stream_wait_event(void *stream, void *event);

/* integer CFA phase: dt_dev_get_roi_filters() develop/imageop.c:139-142 ->
 * dt_rawspeed_crop_dcraw_filters() imageio/imageio_rawspeed.cc:146-151 ->
 * ColorFilterArray::shiftDcrawFilter() external/rawspeed/.../ColorFilterArray.cpp:143-170 */
uint32_t b200_roi_filters(uint32_t filters, int roi_x, int roi_y);
/* FC(), develop/imageop_math.h:190-193 */
int b200_fc(int row, int col, uint32_t filters);

/* ---- demosaic (src/iop/demosaic.c) -------------------------------------------------------- */
/* dt_iop_demosaic_method_t values used here, iop/demosaic.c:109-135 */
enum
{
  B200_DEMOSAIC_PPG = 0,
  B200_DEMOSAIC_AMAZE = 1,
  B200_DEMOSAIC_VNG4 = 2,
  B200_DEMOSAIC_RCD = 5,
  B200_DEMOSAIC_LMMSE = 6
};
/* dt_iop_demosaic_data_t, iop/demosaic.c:238-247 (identical layout) */
typedef struct b200_demosaic_data_t
{
  uint32_t green_eq;
  uint32_t color_smoothing;
  uint32_t demosaicing_method;
  uint32_t lmmse_refine;
  float median_thrs;
  double CAM_to_RGB[3][4];
  float dual_thrs;
} b200_demosaic_data_t;

#define B200_DEMOSAIC_DUAL 2048 /* DEMOSAIC_DUAL, iop/demosaic.c:109: or-ed into the method */
/* process(), iop/demosaic.c:1043-1253: in = 1-channel float mosaic roi_in, out = RGBA float roi_out.  Built for Bayer
 * sensors: RCD (iop/demosaic/rcd.c), AMaZE (amaze.cc), LMMSE (lmmse.c; data->lmmse_refine; every tile from zeroed planes, where the
 * reference carries them from tile to tile: DESIGN.md row f12), PPG with its optional pre-median (ppg.c, basic.c:136-186;
 * data->median_thrs), VNG4 (vng.c, basic.c lin_interpolate), the dual demosaic RCD|DUAL and AMaZE|DUAL (dual.c: blend with
 * VNG4 under the detail mask of develop/masks/detail.c; data->dual_thrs, piece->wb_coeffs), green equilibration in front
 * (data->green_eq) and median colour smoothing behind (data->color_smoothing); the two passthrough methods (3 monochrome,
 * 4 photosite colour; passthrough.c) for any sensor; for X-Trans sensors (filters == 9, piece->xtrans) Markesteijn with one pass
 * (method 1025, the default of X-Trans frames; markesteijn.c:47-521) or three (method 1026) and VNG (method 1024, the X-Trans branch of vng.c); the
 * half-size downsample (method 7, iop/demosaic.c:480-532 Bayer, :543-666 X-Trans; roi_out =
 * (roi_in + 1) / 2; four-colour Bayer sensors through data->CAM_to_RGB) and its guided-Laplacian post-filter (:681-926;
 * data->color_smoothing iterations).  FDC, Markesteijn 3-pass + VNG, the full-size demosaicers on four-colour Bayer sensors and
 * the GUI's mask display return B200_ERR_UNSUPPORTED. */
int b200_demosaic_process_host(const b200_piece_t *piece, const void *in, void *out);
/* process_cl() slot, iop/demosaic/rcd.c:568-850: device pointers, `stream` is a cudaStream_t (NULL = default) */
int b200_demosaic_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
/* tiling_callback(), iop/demosaic.c:1916-2013 */
void b200_demosaic_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- colorin / colorout (src/iop/colorin.c, src/iop/colorout.c) ----------------------------- */
#define B200_LUT_SAMPLES 0x10000 /* DT_CONVERSION_LUT_SAMPLES, colorprofiles/conversion.h:67 */
#define B200_COLORSPACE_LAB 6    /* DT_COLORSPACE_LAB, colorprofiles/profile_types.h:179 */
#define B200_DISPLAY_MASK 1      /* DT_DEV_PIXELPIPE_DISPLAY_MASK bit of pipe->mask_display */

/* How multiply-adds are rounded.  CONTRACT reproduces the reference's release build on an
 * FMA-capable x86-64 (-ffp-contract=fast, gcc 13; pinned bit-for-bit against that build);
 * STRICT is the same source under plain C semantics (-ffp-contract=off). */
enum
{
  B200_FP_CONTRACT = 0,
  B200_FP_STRICT = 1
};

/* What a device kernel needs from dt_colorspaces_conversion_t (colorprofiles/conversion.c:58-97);
 * upstream hands these out through dt_colorspaces_conversion_{is_matrix,has_clipping,matrix,
 * clip_matrix,source_curve,target_curve,source_coeffs,target_coeffs,identity}()
 * (conversion.c:503-506,770-830).  Curves are HOST pointers to B200_LUT_SAMPLES floats (NULL =
 * no curve stage on that side; first entry < 0 = that channel is linear); the library keeps a
 * device copy keyed by `identity`. */
typedef struct b200_conversion_t
{
  int is_matrix;           /* 0 = lcms2 transform: not built here (B200_ERR_UNSUPPORTED) */
  int has_clipping;
  float matrix[3][4];      /* dt_colormatrix_t rows: source -> target, or source -> clip when clipping */
  float clip_matrix[3][4]; /* clip -> target */
  const float *lut_source[3];
  float coeffs_source[3][3]; /* {a, b, c} of b * (a x)^c past white, iop_profile.h:559-562 */
  const float *lut_target[3];
  float coeffs_target[3][3];
  uint64_t identity;       /* 0 = do not cache the curves on the device */
  int fp_mode;             /* B200_FP_CONTRACT (default) or B200_FP_STRICT */
} b200_conversion_t;

/* the fields of dt_iop_colorin_data_t (iop/colorin.c:145-163) that process() reads */
typedef struct b200_colorin_data_t
{
  const b200_conversion_t *conversion; /* NULL = passthrough (colorin.c:720-723) */
  int type;                            /* B200_COLORSPACE_LAB = passthrough */
  int blue_mapping;                    /* legacy hook (colorin.c:690-709): not built, must be 0 */
} b200_colorin_data_t;

/* the fields of dt_iop_colorout_data_t (iop/colorout.c:94-113) that process() reads */
typedef struct b200_colorout_data_t
{
  const b200_conversion_t *conversion;
  int type;
} b200_colorout_data_t;

/* process(), iop/colorin.c:711-734 / iop/colorout.c:373-389: RGBA float in -> RGBA float out, roi_out sized */
int b200_colorin_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_colorin_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
int b200_colorout_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_colorout_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
/* default_tiling_callback(), develop/tiling.c:1423-1463: factor 2, no overlap */
void b200_colorin_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);
void b200_colorout_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);
/* dt_colorspaces_apply_conversion(), colorprofiles/conversion.c:762-766, on device buffers */
int b200_apply_conversion_dev(const b200_conversion_t *conversion, const void *d_in, void *d_out, size_t width,
                              size_t height, int copy_alpha, void *stream);
/* dt_ioppr_init_unbounded_coeffs(), colorprofiles/iop_profile.c:303-329: fit {a,b,c} per channel from a
 * 3 x B200_LUT_SAMPLES curve set (host side, called from commit_params); returns the number of
 * non-linear channels */
int b200_fit_unbounded_coeffs(const float *const lut[3], float coeffs[3][3]);

/* ---- denoise (profiled) (src/iop/denoiseprofile.c) ------------------------------------------------ */
#define B200_DENOISE_BANDS 7 /* DT_IOP_DENOISE_PROFILE_BANDS, denoiseprofile.c:109 */
enum
{ /* dt_iop_denoiseprofile_mode_t, denoiseprofile.c:120-126 */
  B200_DENOISE_NLMEANS = 0,
  B200_DENOISE_WAVELETS = 1,
  B200_DENOISE_VARIANCE = 2,
  B200_DENOISE_NLMEANS_AUTO = 3,
  B200_DENOISE_WAVELETS_AUTO = 4
};
enum
{ /* dt_iop_denoiseprofile_wavelet_mode_t :128-131 and dt_iop_denoiseprofile_channel_t :134-143 */
  B200_DENOISE_RGB = 0,
  B200_DENOISE_Y0U0V0 = 1,
  B200_DENOISE_CH_ALL = 0,
  B200_DENOISE_CH_R = 1,
  B200_DENOISE_CH_G = 2,
  B200_DENOISE_CH_B = 3,
  B200_DENOISE_CH_Y0 = 4,
  B200_DENOISE_CH_U0V0 = 5,
  B200_DENOISE_CH_NONE = 6
};
/* The members of dt_iop_denoiseprofile_data_t (denoiseprofile.c:352-371) that process() reads, same
 * names and meaning; the GUI curve handles of the reference struct are dropped, `force` is what
 * commit_params evaluates from them (:2864-2872). */
typedef struct b200_denoiseprofile_data_t
{
  float radius, nbhood, strength, shadows, bias, scattering, central_pixel_weight, overshooting;
  float a[3], b[3];
  int mode;
  float force[B200_DENOISE_CH_NONE][B200_DENOISE_BANDS];
  int wb_adaptive_anscombe, fix_anscombe_and_nlmeans_norm, use_new_vst;
  int wavelet_color_mode;
} b200_denoiseprofile_data_t;

/* process(), denoiseprofile.c:2633-2647 -> process_wavelets :1289-1447 / process_nlmeans :1599-1654 */
int b200_denoiseprofile_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_denoiseprofile_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
/* tiling_callback(), denoiseprofile.c:796-849 */
void b200_denoiseprofile_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);
/* the two wavelet kernels on their own (pixel/eaw.c:242-326, :157-175): device RGBA buffers.
 * d_sum_squared receives 4 doubles (sum over pixels of detail^2 per channel). */
int b200_eaw_dn_decompose_dev(void *d_coarse, const void *d_in, void *d_detail, double *d_sum_squared, int scale,
                              float inv_sigma2, int width, int height, void *stream);
int b200_eaw_synthesize_dev(void *d_out, const void *d_in, const void *d_detail, const float threshold[4],
                            const float boost[4], int width, int height, void *stream);
/* nlmeans_denoise(), pixel/nlmeans_core.c:315-532 (dt_nlmeans_param_t spelled out): device RGBA buffers,
 * d_in != d_out.  center_weight < 0 selects the denoise (non-local means) iop's weighting (:389-402),
 * >= 0 the profiled one (:404-420).  Patch radius 0..4. */
int b200_nlmeans_denoise_dev(const void *d_in, void *d_out, int width, int height, float scattering, float scale, float luma,
                             float chroma, float center_weight, float sharpness, int patch_radius, int search_radius,
                             int decimate, const float norm[4], void *stream);

/* ---- filmic rgb (src/iop/filmicrgb.c) ---------------------------------------------------------- */
/* dt_iop_filmic_rgb_spline_t, filmicrgb.c:216-223 (identical layout, 144 bytes) */
typedef struct b200_filmic_spline_t
{
  float M1[4] __attribute__((aligned(16)));
  float M2[4] __attribute__((aligned(16)));
  float M3[4] __attribute__((aligned(16)));
  float M4[4] __attribute__((aligned(16)));
  float M5[4] __attribute__((aligned(16)));
  float latitude_min, latitude_max;
  float y[5];
  float x[5];
  int type[2]; /* dt_iop_filmicrgb_curve_type_t: 0 poly4, 1 poly3, 2 rational, 3 sigmoid */
} b200_filmic_spline_t;

/* dt_iop_filmicrgb_data_t, filmicrgb.c:360-400 (identical layout, 832 bytes): what commit_params()
 * :4005-4113 leaves in piece->data is passed through unchanged */
typedef struct b200_filmicrgb_data_t
{
  float max_grad, white_source, grey_source, black_source;
  float reconstruct_threshold, reconstruct_feather, reconstruct_bloom_vs_details, reconstruct_grey_vs_color,
      reconstruct_structure_vs_texture;
  float normalize, dynamic_range, saturation, output_power, contrast, sigma_toe, sigma_shoulder, noise_level;
  int preserve_color;
  int version; /* dt_iop_filmicrgb_colorscience_type_t: 0..4 = "v3 (2019)".."v7 (2023)", 5..9 = the AgX (v8) family */
  int spline_version;
  int high_quality_reconstruction;
  int hl_deprecated;
  float agx_beta_hue;
  b200_filmic_spline_t spline __attribute__((aligned(64)));
  int noise_distribution;
  int softproof_mode, softproof_type;
  char softproof_filename[512];
  int softproof_intent;
} b200_filmicrgb_data_t;

/* RGB <-> XYZ(D50) of a matrix profile: dt_iop_order_iccprofile_info_t.matrix_in / matrix_out
 * (colorprofiles/iop_profile.h:127-131), rows of a dt_colormatrix_t */
typedef struct b200_profile_matrices_t
{
  float matrix_in[3][4];
  float matrix_out[3][4];
} b200_profile_matrices_t;

/* what filmic's process() reads: piece->data plus the two pipe-level profiles it fetches through
 * dt_ioppr_get_pipe_work_profile_info() and _filmic_get_output_profile() (filmicrgb.c:2714-2715) */
typedef struct b200_filmicrgb_piece_t
{
  b200_filmicrgb_data_t data;
  b200_profile_matrices_t work_profile;
  int has_export_profile;          /* 0 = output profile is not a matrix profile: gamut-map in the work space */
  b200_profile_matrices_t export_profile;
} b200_filmicrgb_piece_t;

/* process(), filmicrgb.c:2707-2895.  Built: every colour science -- the AgX family (version 5..9, :2495-2587) and the
 * earlier ones (0..4: filmic_split/chroma_v1, _v2_v3, _v4, filmic_v5, :1534-1737,2153-2299) with any chroma-preservation
 * norm -- and, for edits that still carry a reconstruction threshold (hl_deprecated == 0; off by default), the wavelet
 * highlight reconstruction in front of them (:1201-1532, 2729-2838; reads piece->buf_in_*, iscale and roi_in.scale
 * for its scale count, and synchronises the stream once to learn whether anything is clipped).  The display of the
 * clipping mask is GUI state and stays in the reference.  A work profile with tone curves is not representable in
 * b200_profile_matrices_t (the luminance norm then needs its LUTs). */
int b200_filmicrgb_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_filmicrgb_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
/* tiling_callback(), filmicrgb.c:2668-2704 */
void b200_filmicrgb_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- local contrast (src/iop/bilat.c): local-Laplacian and bilateral-grid modes ------------------ */
enum
{ /* dt_iop_bilat_mode_t, bilat.c:71-76 */
  B200_BILAT_BILATERAL = 0,
  B200_BILAT_LOCAL_LAPLACIAN = 1
};
/* dt_iop_bilat_data_t == dt_iop_bilat_params_t, bilat.c:78-86,108 (identical layout) */
typedef struct b200_bilat_data_t
{
  int mode;      /* default 1 */
  float sigma_r; /* highlights, default 0.5 */
  float sigma_s; /* shadows, default 0.5 */
  float detail;  /* clarity, default 0.25 */
  float midtone; /* default 0.5 */
} b200_bilat_data_t;
/* process(), bilat.c:336-360.  Mode 1 -> local_laplacian_internal(), pixel/locallaplacian.c:354-563.  Mode 0 -> the bilateral
 * grid of pixel/bilateral.c (init, splat, blur, slice :157-393) with sigma_s divided by the module scale (piece->iscale /
 * roi_in.scale); the reference's splat rounds differently for different OpenMP thread counts (one horizontal slice per
 * thread, partial grids added afterwards): the result here is the one-slice, raster-order one.  Lab RGBA in/out;
 * channels 1,2 are copied, channel 3 carried through from the input. */
int b200_bilat_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_bilat_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_bilat_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- diffuse or sharpen (src/iop/diffuse.c) ----------------------------------------------------- */
#define B200_DIFFUSE_MAX_SCALES 10 /* MAX_NUM_SCALES, diffuse.c:75 */
/* dt_iop_diffuse_data_t == dt_iop_diffuse_params_t, diffuse.c:76-109,132 (identical layout, 60 bytes) */
typedef struct b200_diffuse_data_t
{
  int iterations;           /* default 1 */
  float sharpness;          /* 0 */
  int radius;               /* 8 */
  float regularization;     /* 0 */
  float variance_threshold; /* 0 */
  float anisotropy_first, anisotropy_second, anisotropy_third, anisotropy_fourth;
  float threshold;          /* luminance masking threshold; > 0: only pixels above it are solved, from a noise-seeded start */
  float first, second, third, fourth;
  int radius_center;
} b200_diffuse_data_t;
/* process(), diffuse.c:1155-1259: iterations x (a-trous B-spline decomposition into `scales` bands, then the
 * anisotropic heat PDE band by band from coarse to fine).  zoom = piece->iscale / roi_in.scale. */
int b200_diffuse_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_diffuse_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
/* tiling_callback(), diffuse.c:585-610 */
void b200_diffuse_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- denoise (non-local means) iop (src/iop/nlmeans.c) ------------------------------------------ */
/* dt_iop_nlmeans_data_t == dt_iop_nlmeans_params_t, nlmeans.c:81-88,98 */
typedef struct b200_nlmeans_data_t
{
  float radius;   /* patch size, default 2 */
  float strength; /* default 50 */
  float luma;     /* default 0.5 */
  float chroma;   /* default 1.0 */
} b200_nlmeans_data_t;
/* process() :458-465 -> process_cpu :416-456 -> nlmeans_denoise() in Lab with center_weight = -1.  The
 * patches are decimated on thumbnail and preview pipes (pipe_type B200_PIPE_THUMBNAIL / B200_PIPE_PREVIEW). */
int b200_nlmeans_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_nlmeans_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
/* tiling_callback(), nlmeans.c:400-414 */
void b200_nlmeans_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- RGB <-> Lab between modules of different colour space ------------------------------------------
 * dt_colorspaces_apply_profile(), colorprofiles/iop_profile.c:1300-1359 -> dt_ioppr_transform_matrix :566-596
 * -> _transform_rgb_to_lab_matrix :376-420 / _transform_lab_to_rgb_matrix :422-464, for the pipe's work
 * profile.  b200_colorspace_transform_dev is the linear-profile call (nonlinearlut == 0: linear Rec2020, the default,
 * and every other "linear ..." built-in; nonlinearlut != 0 is refused there); a work profile with tone curves goes
 * through b200_colorspace_transform_trc_dev with its curves (_apply_tonecurves :332-373).
 * cst: dt_iop_colorspace_type_t (pixel/format.h): 1 = IOP_CS_LAB, 2 = IOP_CS_RGB.  d_in == d_out allowed.
 * RGB -> Lab leaves lane 3 as the reference does (not written: in place it keeps the pixel's alpha, which is
 * what this entry stores); Lab -> RGB copies the input alpha. */
#define B200_CS_LAB 1
#define B200_CS_RGB 2
int b200_colorspace_transform_dev(const void *d_in, void *d_out, int width, int height, int cst_from, int cst_to,
                                  const b200_profile_matrices_t *work_profile, int nonlinearlut, void *stream);
/* Tone curves of a matrix profile, dt_iop_order_iccprofile_info_t (colorprofiles/iop_profile.h:137-156): lut_in /
 * lut_out are host arrays of B200_LUT_SAMPLES floats (lutsize 65536, the only size the reference uses), lut[k][0] < 0
 * marks channel k linear; unbounded_coeffs_* are the {a, b, c} of b * (a x)^c past 1.0.  As in the reference the
 * profile counts as non-linear by its INPUT curves alone (dt_ioppr_init_unbounded_coeffs, iop_profile.c:303-329):
 * with three linear lut_in the call equals the linear one whatever lut_out holds.  RGB -> Lab: a channel without a
 * curve and lane 3 keep the pixel's values (the reference's in-place behaviour).  identity != 0 caches the device
 * copy of the curves. */
typedef struct b200_profile_curves_t
{
  const float *lut_in[3];
  const float *lut_out[3];
  float unbounded_coeffs_in[3][3];
  float unbounded_coeffs_out[3][3];
  uint64_t identity;
} b200_profile_curves_t;
int b200_colorspace_transform_trc_dev(const void *d_in, void *d_out, int width, int height, int cst_from, int cst_to,
                                      const b200_profile_matrices_t *work_profile, const b200_profile_curves_t *curves, void *stream);

/* ---- sharding one frame over several GPUs (SURVEY.md 8e) ---------------------------------------
 * Row bands = full-width tiles of the reference's tiling engine (src/develop/tiling.c:723-1075).
 * A band reads input rows [in_y0,in_y1) with roi_in.y = in_y0 and owns output rows [out_y0,out_y1). */
#define B200_MAX_BANDS 64
typedef struct b200_band_t
{
  int out_y0, out_y1;
  int in_y0, in_y1;
} b200_band_t;
/* grid == 1: cuts at multiples of `align`, `halo` rows of overlap on both sides (the tiling_callback numbers,
 * summed over the chained modules).  grid > 1: cuts at k*grid+halo so a module with an internal block grid
 * (RCD: grid 94, halo 9) gives the same bits as on the untiled frame.  Bands may come out empty when
 * n_bands exceeds the number of block rows. */
int b200_band_plan(int height, int n_bands, int grid, int halo, int align, b200_band_t *bands);
/* The gather fused into the producing kernel: the last (pointwise) module of a band stores every result pixel
 * into up to B200_MAX_SCATTER frames -- this GPU's and, through peer mappings, the other GPUs' -- so the
 * exchange rides on the kernel's own stores over NVLink instead of following it as a collective.
 * d_outs[k] points at the band's first output row inside frame k.  Peer frames are mapped with the IPC calls
 * below (one process per GPU); the caller separates the stores from the consumers with a stream
 * synchronisation and a barrier across the processes. */
#define B200_MAX_SCATTER 8
int b200_apply_conversion_scatter_dev(const b200_conversion_t *conv, const void *d_in, int n_out, void *const *d_outs,
                                      size_t width, size_t height, int copy_alpha, void *stream);
int b200_colorout_process_scatter_dev(const b200_piece_t *piece, const void *d_in, int n_out, void *const *d_outs, void *stream);
/* cudaIpcGetMemHandle / OpenMemHandle / CloseMemHandle on a b200_dev_alloc() allocation; handle = 64 opaque bytes */
#define B200_IPC_HANDLE_BYTES 64
int b200_ipc_export(void *d_ptr, unsigned char handle[B200_IPC_HANDLE_BYTES]);
int b200_ipc_import(const unsigned char handle[B200_IPC_HANDLE_BYTES], void **d_ptr);
int b200_ipc_release(void *d_ptr);
/* Row grid, halo and alignment for b200_band_plan() under which a banded demosaic equals the untiled frame bit
 * for bit: RCD's 94-row blocks with a 9-row halo (rcd.c:71-75).  AMaZE mirrors the frame edge at its own tile
 * origin (amaze.cc:357-455), so no cut reproduces the untiled frame: grid 1 and the tiling_callback() overlap
 * (demosaic.c:1916-2013) come back, i.e. bands are tiles of develop/tiling.c.  piece == NULL means RCD. */
void b200_demosaic_band_grid(const b200_piece_t *piece, int *grid, int *halo, int *align);

/* ==== the modules either side of the demosaic .. colorout path (SURVEY.md section 8f, ranks 1 and 2) ============ */

/* ---- rawprepare (src/iop/rawprepare.c): sensor data -> normalised float mosaic ------------------------------- */
/* dt_dng_gain_map_t, src/common/dng_opcode.h:37-55 (identical layout; host memory) */
typedef struct b200_dng_gain_map_t
{
  uint32_t top, left, bottom, right, plane, planes, row_pitch, col_pitch;
  uint32_t map_points_v, map_points_h;
  double map_spacing_v, map_spacing_h, map_origin_v, map_origin_h;
  uint32_t map_planes;
  float map_gain[];
} b200_dng_gain_map_t;
/* dt_iop_rawprepare_data_t, rawprepare.c:94-111 (identical layout) */
typedef struct b200_rawprepare_data_t
{
  int32_t x, y, width, height; /* sensor border trim */
  float sub[4];                /* black level per CFA site of the 2x2 block */
  float div[4];                /* white - black */
  struct
  {
    uint16_t raw_black_level, raw_white_point;
  } rawprepare;
  int apply_gainmaps;
  b200_dng_gain_map_t *gainmaps[4]; /* one per site of the RGGB block when apply_gainmaps */
} b200_rawprepare_data_t;
/* process() :466-633.  Input: roi_in.width x roi_in.height samples of piece->datatype (uint16 or float mosaic when
 * piece->filters != 0 and channels == 1, else `channels` floats per pixel); output roi_out floats.  Gain maps are
 * bilinearly interpolated per site (:592-630).  process_cl() :636-760 is the same arithmetic. */
int b200_rawprepare_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_rawprepare_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_rawprepare_tiling(const b200_piece_t *piece, b200_tiling_t *tiling); /* default_tiling_callback, imageop.c */

/* ---- temperature (src/iop/temperature.c): white-balance multipliers ---------------------------------------------- */
/* dt_iop_temperature_data_t, temperature.c:150-153 */
typedef struct b200_temperature_data_t
{
  float coeffs[4];
} b200_temperature_data_t;
/* process() :486-608: Bayer mosaic (coefficient by FC at roi_out origin), X-Trans mosaic (FCxtrans), or `channels`
 * floats per pixel (alpha carried; copied from the input when a mask is displayed) */
int b200_temperature_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_temperature_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_temperature_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- highlights (src/iop/highlights.c): clip mode + the "nothing to reconstruct" bypass -------------------------- */
enum
{
  B200_HIGHLIGHTS_CLIP = 0,
  B200_HIGHLIGHTS_LCH = 1,
  B200_HIGHLIGHTS_INPAINT = 2,
  B200_HIGHLIGHTS_LAPLACIAN = 3,
  B200_HIGHLIGHTS_HARMONIC = 4
};
/* dt_iop_highlights_data_t == dt_iop_highlights_params_t, iop/highlights/common.h:456-476 (identical layout) */
typedef struct b200_highlights_data_t
{
  int mode;
  float blendL, blendC, blendh;
  float clip;
  float noise_level;
  int iterations;
  int scales;
  float reconstructing;
  float combine;
  int debugmode;
  float solid_color;
} b200_highlights_data_t;
/* process() :679-789: counts the samples above the mode's threshold (_hl_count_clipped :266-292); fewer than 25 ->
 * the input is copied through.  Past the bypass, built: mode CLIP (process_clip, iop/highlights/clip.c:60-85; also
 * what LCh and colour inpainting run on non-mosaic input) and, on Bayer and X-Trans mosaics alike, LCh (process_lch_bayer /
 * process_lch_xtrans, iop/highlights/lch.c:315-537; their long-double products, quotients and sums in integer arithmetic,
 * x87.cuh) and colour inpainting (process_inpaint_bayer / _xtrans, iop/highlights/inpaint.c:63-104: four directional line
 * recurrences, averaged).  For these the count and the branch stay on the device: no host round trip.  Guided Laplacians
 * (below) run once the host has read the count; harmonic transposition returns B200_ERR_UNSUPPORTED
 * when the frame does not take the bypass. */
/* Mode LAPLACIAN past the bypass (process_laplacian, iop/highlights/laplacian.c:433-575) on a Bayer or X-Trans mosaic or on RGBA input: the
 * frame gathered into [R, G, B, norm] and a clipping mask (iop/highlights/gather.c), the mask feathered by a box mean, both reduced
 * to a quarter, `iterations` rounds of guide_laplacians and heat_PDE_diffusion over the wavelet scales, enlarged and composited.
 * `normalization`: NULL in production.  The reference's vector (_compute_laplacian_normalization, gather.c:223-275) is an OpenMP
 * float reduction whose value depends on the thread count; the library sums in double in a fixed order.  A caller that has the
 * vector of one reference run (4 floats, host memory) passes it and gets that run's bits.  No bypass test here: the frame is
 * reconstructed whatever its count.  Frames under 8 px either way: B200_ERR_UNSUPPORTED (the reference's quarter-size planes vanish). */
int b200_highlights_laplacian_dev(const b200_piece_t *piece, const void *d_in, void *d_out, const float *normalization, void *stream);
int b200_highlights_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_highlights_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_highlights_tiling(const b200_piece_t *piece, b200_tiling_t *tiling); /* :575-644 */

/* ---- the three of them in one pass over the sensor data (pipe-level fusion) ---------------------------------------
 * What rawprepare -> temperature -> highlights(clip) compute on a Bayer mosaic, sample by sample in the same order
 * and precision, without the two intermediate float planes: bit-identical to calling the three entry points one
 * after the other (tests/test_zz_pipe_ends_gpu.py).  pieces: [0] rawprepare's, [1] temperature's, [2] highlights'
 * (NULL = module disabled).  26 -> 8 bytes per sample of HBM traffic for uint16 input. */
int b200_rawfront_process_dev(const b200_piece_t *rawprepare, const b200_piece_t *temperature, const b200_piece_t *highlights,
                              const void *d_in, void *d_out, void *stream);

/* ---- exposure (src/iop/exposure.c) ------------------------------------------------------------------------------- */
/* dt_iop_exposure_data_t, exposure.c:151-157 with dt_iop_exposure_params_t :116-124 (identical layout) */
typedef struct b200_exposure_data_t
{
  struct
  {
    int mode;
    float black, exposure, deflicker_percentile, deflicker_target_level;
    int compensate_exposure_bias;
  } params;
  int deflicker;
  float black; /* as _process_common_setup() :433-470 left them */
  float scale;
} b200_exposure_data_t;
/* process() :501-544: (in - black) * scale on every float of the pixel (alpha included when channels == 4) */
int b200_exposure_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_exposure_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_exposure_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- colour calibration (src/iop/channelmixerrgb.c) ------------------------------------------------------------ */
/* dt_adaptation_t, src/pixel/chromatic_adaptation.h:34-42 (same values) */
enum
{
  B200_ADAPTATION_LINEAR_BRADFORD = 0,
  B200_ADAPTATION_CAT16 = 1,
  B200_ADAPTATION_FULL_BRADFORD = 2,
  B200_ADAPTATION_XYZ = 3,
  B200_ADAPTATION_RGB = 4
};
/* dt_iop_channelmixer_rbg_data_t, channelmixerrgb.c:259-272 (identical layout: 64-byte aligned, 192 bytes) */
typedef struct b200_channelmixerrgb_data_t
{
  float MIX[4][4] __attribute__((aligned(64))); /* dt_colormatrix_t: the 3x3 channel mix, rows padded to 4 */
  float saturation[4] __attribute__((aligned(16)));
  float lightness[4] __attribute__((aligned(16)));
  float grey[4] __attribute__((aligned(16)));
  float illuminant[4] __attribute__((aligned(16))); /* in the adaptation's LMS (or XYZ) space */
  float p, gamut;
  int apply_grey;
  int clip;
  int adaptation;      /* B200_ADAPTATION_* */
  int illuminant_type; /* dt_illuminant_t; read by the reference's process() before the pixel loop, not by the library */
  int version;         /* dt_iop_channelmixer_rgb_version_t: 0 (2020), 1 (2021), 2 (Apr 2021) */
} b200_channelmixerrgb_data_t;
/* what the pixel loop reads: piece->data plus the work profile's matrices process() fetches (:1926, :1936-1942) */
typedef struct b200_channelmixerrgb_piece_t
{
  b200_channelmixerrgb_data_t data;
  b200_profile_matrices_t work_profile;
} b200_channelmixerrgb_piece_t;
/* process() :1920-2078 from the switch on data->adaptation on: loop_switch() :765-959 = chromatic adaptation (Bradford
 * linear / full, CAT16, XYZ, none) + channel mix + gamut compression in xyY/uvY (gamut_mapping :641-706) + the
 * colourfulness / brightness adjustment (luma_chroma :707-763) + optional grey output, with every clip of the reference.
 * What precedes the switch stays the reference's C: the GUI's colour-checker fit and illuminant detection, and the
 * re-derivation of data->illuminant for the "as shot in camera" illuminant from the image metadata (:1986-2014). */
int b200_channelmixerrgb_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_channelmixerrgb_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_channelmixerrgb_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- finalscale (src/iop/finalscale.c): the export's final resampling ------------------------------------------- */
/* enum dt_interpolation_type, src/pixel/interpolation.h:38-44 (same values) */
enum
{
  B200_INTERPOLATION_BILINEAR = 0,
  B200_INTERPOLATION_BICUBIC = 1,
  B200_INTERPOLATION_MITCHELL = 2 /* DT_INTERPOLATION_DEFAULT */
};
/* dt_iop_finalscale_data_t (finalscale.c:46-51: one dummy int) + the interpolator process() resolves from the user
 * preference (dt_interpolation_new(DT_INTERPOLATION_USERPREF), plugins/lighttable/export/pixel_interpolator): the
 * adapter passes its id, the library reads no configuration */
typedef struct b200_finalscale_data_t
{
  int dummy;
  int interpolator; /* B200_INTERPOLATION_* */
} b200_finalscale_data_t;
/* process() :117-131 = dt_iop_clip_and_zoom_roi -> _interpolation_resample_plain (pixel/interpolation.c:897-1027) with
 * both ROI origins zeroed: roi_in.width x height RGBA at roi_in.scale -> roi_out.width x height at roi_out.scale.  The
 * two per-axis tap plans (_prepare_resampling_plan :710-893) are built on the host as in the reference; every output
 * pixel accumulates its taps in the reference's order (rows, then columns within a row), negative and non-finite
 * results become 0.  Equal scales (or roi_out.scale == 1) copy rows. */
int b200_finalscale_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_finalscale_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_finalscale_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);
/* One axis of the plan, for inspection (lengths[out], kernel/index concatenated, at most max_taps): returns the number of
 * taps, -1 for scale == 1 (no resampling), < -1 on error */
int b200_resampling_plan(int interpolator, int in, int in_x0, int out, int out_x0, float scale, int *lengths, float *kernel, int *index,
                         int max_taps);

/* ---- basebuffer (src/iop/basebuffer.c): the pipe's first node, sensor buffer -> first cacheline ------------------------- */
/* process() :119-160 copies the crop roi_out out of the full-size buffer the mipmap cache holds (host memory, pipe->iwidth x
 * pipe->iheight samples of dsc_in.bpp bytes) into the module's output.  On the device that copy IS the upload: one strided
 * host-to-device transfer into the device cacheline, nothing else touches the bytes.  bpp: piece->dsc_in.bpp (2 for uint16
 * sensor data, 4 for float mosaics, 16 for float RGBA).  Rows or columns of roi_out beyond the buffer are left as found, as
 * in the reference (:133-134). */
int b200_basebuffer_upload_dev(const b200_piece_t *piece, const void *host_full, int iwidth, int iheight, size_t bpp, void *d_out, void *stream);

/* ---- initialscale (src/iop/initialscale.c): the darkroom's first resampling ---------------------------------------- */
/* process() :122-129 = dt_iop_clip_and_zoom_roi with both ROIs as they are: the resampler of finalscale with the ROI origins in
 * its tap plans (and, between equal scales, a crop at roi_out - roi_in).  piece->data: a b200_finalscale_data_t (the module's
 * own data block is a dummy int; the interpolator is the user preference the adapter resolves). */
int b200_initialscale_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_initialscale_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_initialscale_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- flip (src/iop/flip.c): orientation ---------------------------------------------------------------------------- */
/* dt_iop_flip_data_t == dt_iop_flip_params_t, flip.c:74-79: dt_image_orientation_t (common/image.h:213-231): bit 0 flip y,
 * bit 1 flip x, bit 2 swap x and y (the output then has roi_in.height columns) */
typedef struct b200_flip_data_t
{
  int orientation;
} b200_flip_data_t;
/* process() :388-400 -> dt_imageio_flip_buffers (imageio/imageio_core.c:258-297) on roi_in.width x roi_in.height pixels of
 * piece->channels floats */
int b200_flip_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_flip_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_flip_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- gamma (src/iop/gamma.c): the pipe's last module, float RGBA -> uint8 BGRA for the display --------------------- */
/* process() :367-377 with no mask or channel display: _copy_output :352-364 (the fourth byte of every output pixel is
 * not written).  Mask and false-colour displays (GUI previews) return B200_ERR_UNSUPPORTED. */
int b200_gamma_process_host(const b200_piece_t *piece, const void *in, void *out);
int b200_gamma_process_dev(const b200_piece_t *piece, const void *d_in, void *d_out, void *stream);
void b200_gamma_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

/* ---- the export's down-conversion of the float backbuffer (src/imageio/imageio_core.c:706-738) ---------------------
 * B200_EXPORT_UINT8 _clamp_float_to_uint8, B200_EXPORT_UINT8_SWAP _swap_byteorder_float_to_uint8 (BGRA),
 * B200_EXPORT_UINT16 _export_final_buffer_to_uint16.  Done on the device, the read-back of a finished frame is 4 or
 * 8 bytes per pixel instead of 16. */
enum
{
  B200_EXPORT_UINT8 = 0,
  B200_EXPORT_UINT8_SWAP = 1,
  B200_EXPORT_UINT16 = 2
};
int b200_export_convert_dev(const void *d_in, void *d_out, size_t width, size_t height, int format, void *stream);
int b200_export_convert_host(const void *in, void *out, size_t width, size_t height, int format);

/* ---- the libm the kernels use ------------------------------------------------------------------
 * Device restatement of glibc 2.39's single-precision expf/exp2f/logf/log2f/powf/sinf/cosf/atanf/atan2f/hypotf (the functions the
 * reference's CPU path calls; see ansel_b200/csrc/flt32_math.cuh).  Exposed so its bit-compatibility
 * with the host libm can be verified on the machine the pipe runs on. */
enum
{
  B200_FLT32_EXPF = 0,
  B200_FLT32_EXP2F = 1,
  B200_FLT32_LOGF = 2,
  B200_FLT32_LOG2F = 3,
  B200_FLT32_POWF = 4,
  B200_FLT32_SINF = 5, /* |x| < 120 */
  B200_FLT32_COSF = 6,
  B200_FLT32_ATANF = 7,
  B200_FLT32_ATAN2F = 8, /* atan2f(x[k], y[k]): x is the ordinate */
  B200_FLT32_HYPOTF = 9
};
int b200_flt32_eval_dev(int fn, const float *d_x, const float *d_y, float *d_out, size_t n, void *stream);

/* ---- blending of a module's output over its input: develop/blend.c dt_develop_blend_process :657-860 --------------------------------
 * The members of dt_develop_blend_params_t (develop/blend.h:197-237, piece->blendop_data) the path reads, under their own names, then
 * what the reference looks up on the host for the same call. */
typedef struct b200_blend_params_t
{
  uint32_t mask_mode;        /* dt_develop_mask_mode_t: 1 enabled, 2 drawn mask, 4 parametric mask, 8 raster mask */
  int32_t blend_cst;         /* dt_develop_blend_colorspace_t: 1 = DEVELOP_BLEND_CS_RAW (buffers of one float per site), 2 = DEVELOP_BLEND_CS_LAB,
                                3 = DEVELOP_BLEND_CS_RGB_DISPLAY, 4 = DEVELOP_BLEND_CS_RGB_SCENE */
  uint32_t blend_mode;       /* dt_develop_blend_mode_t, | 0x80000000 = DEVELOP_BLEND_REVERSE */
  float blend_parameter;     /* exposure-like parameter of the operator, in EV */
  float opacity;             /* 0 .. 100 */
  uint32_t mask_combine;     /* dt_develop_mask_combine_mode_t: 1 inverted, 2 inclusive */
  uint32_t blendif;          /* dt_develop_blendif_channels_t: bits 0..3 / 4..7 gray, red, green, blue (Lab: L, a, b), bits 8..10 / 12..14 Jz, Cz, hz (display
                                RGB: H, S, L; Lab: chroma, hue) of the input / output take part; bit + 16: that channel inverted */
  float feathering_radius;
  uint32_t feathering_guide;
  float blur_radius, contrast, brightness, details;
  float blendif_parameters[64];    /* four limits per channel */
  float blendif_boost_factors[16];
  int32_t raster_used, drawn_used; /* dt_develop_blend_get_mask_usage() :262-320: the form mask passed is a raster mask / a drawn mask (or their
                                      combination, _develop_blend_combine_masks :593-601) */
  float luminance[3];              /* row Y of matrix_in of the pipe's current profile (dt_ioppr_get_rgb_matrix_luminance, iop_profile.h:637-654) */
  int32_t profile_nonlinear;       /* that profile's nonlinearlut: must be 0 */
  uint32_t mask_display;           /* pipe->mask_display: with B200_DISPLAY_MASK the alpha lane of the input is kept (:952-961) */
  float matrix_in[9];              /* that profile's matrix_in (RGB -> XYZ D50), row by row: what the Jz / Cz / hz channels of the parametric mask start
                                      from (dt_develop_blendif_init_masking_profile, develop/blend.c:322-353); read only when bits 8..10 / 12..14 of
                                      `blendif` are set in the RGB space */
} b200_blend_params_t;
/* in: the module's input (roi_in, RGBA float), out: the module's output (roi_out, inside roi_in), blended in place with the mask in its
 * alpha lane (no alpha lane in the raw space); form_mask: the raster / drawn mask of roi_out the host rasterised, or NULL; mask: receives the final mask (what the reference
 * publishes as the module's raster mask, :892-950), or NULL.  Built: the scene-referred RGB space (develop/blends/blendif_rgb_jzczhz.c) with
 * uniform, raster, drawn and parametric (gray, red, green, blue, Jz, Cz, hz of input and output) masks, their exclusive / inclusive / inverted
 * combinations, the mask tone curve and the sixteen blend operators; the Lab space (develop/blends/blendif_lab.c, what local contrast and the
 * other Lab modules blend in) with the same masks on the L, a, b, chroma and hue channels and its twenty-six operators; the display-referred
 * RGB space (develop/blends/blendif_rgb_hsl.c) with the gray, red, green, blue, H, S, L channels and its twenty-seven operators.
 * The raw space (develop/blends/blendif_raw.c): `in` and `out` hold one float per site, uniform / raster / drawn masks, sixteen operators.
 * B200_ERR_UNSUPPORTED (fall back to dt_develop_blend_process): feathering, blur and detail refinement of the mask.  mask_mode without the enabled bit: B200_OK, nothing touched. */
int b200_blend_process_host(const b200_piece_t *piece, const b200_blend_params_t *bp, const void *in, void *out, const float *form_mask, float *mask);
/* dt_develop_blend_process_cl() slot, develop/blend.c:1113-1604: device pointers */
int b200_blend_process_dev(const b200_piece_t *piece, const b200_blend_params_t *bp, const void *d_in, void *d_out, const float *d_form_mask,
                           float *d_mask, void *stream);
/* tiling_callback_blendop(), develop/blend.c:1672-1691 */
void b200_blend_tiling(const b200_piece_t *piece, b200_tiling_t *tiling);

#ifdef __cplusplus
}
#endif
#endif /* B200IOP_H */
