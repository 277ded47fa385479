/*
 * uwip.h - C ABI of libuwip.so: the B200 (sm_100a) implementation of uwimageproc's per-frame
 * enhancement chain  histretch -> aclahe -> bgdehaze.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  Every entry point names the reference interface it
 * replaces (paths relative to the reference tree).  Plain C: pointers, sizes, explicit parameters,
 * an opaque context and an int status.  No OpenCV / numpy / torch types.
 *
 * Conventions
 *   - Frames are 8-bit, 3 interleaved channels in OpenCV order B,G,R ("bgr8"); planes are 8-bit
 *     single channel ("u8").  `pitch` is the byte distance between rows (>= width*channels).
 *   - Functions without a suffix take HOST pointers: they stage through the context's device
 *     workspace on the context's stream and return after the result is back in host memory.
 *   - Functions ending in `_dev` take DEVICE pointers (contiguous rows: pitch == width*channels),
 *     are stream ordered on the context's stream and do NOT synchronise.
 *   - Return value: UWIP_OK (0) or a negative uwip_status; uwip_last_error() gives the text.
 *     The reference prints and continues ("not recognized, skipping", histretch.cpp:252) or has
 *     undefined behaviour (preprocessing.h:60-64); across an ABI those become status codes.
 *   - Threading: a context is single-owner (one context per host thread and device); all work of a
 *     context is ordered on its stream; there is no hidden global state.
 *   - There is no CPU fallback: every entry point fails with UWIP_ERR_CUDA when no sm_100 device
 *     is usable.
 */
#ifndef UWIP_H
#define UWIP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UWIP_VERSION 100

typedef enum uwip_status {
  UWIP_OK = 0,
  UWIP_ERR_INVALID = -1,     /* bad pointer / size / parameter (reference: UB or silent skip)   */
  UWIP_ERR_CUDA = -2,        /* CUDA runtime error, text in uwip_last_error                     */
  UWIP_ERR_UNSUPPORTED = -3, /* valid input this build does not handle: JPEG codings uwip_jpeg_decode_bgr8_batch refuses */
  UWIP_ERR_NOMEM = -4
} uwip_status;

/* HSV->BGR rounding rule of the OpenCV build being replaced (SURVEY appendix A.3). */
typedef enum uwip_hsv_round {
  UWIP_HSV_ROUND_CV2_4_13 = 0, /* trunc for x < 32*floor(W/32), rint for the row tail (cv2 4.13.0 here) */
  UWIP_HSV_ROUND_TRUNC = 1,
  UWIP_HSV_ROUND_RINT = 2      /* documented OpenCV 3.4.6 behaviour */
} uwip_hsv_round;

/* histretch CLI channel-loop order (histretch.cpp:232-240). */
typedef enum uwip_order {
  UWIP_ORDER_INTENDED = 0, /* convert -> stretch -> merge -> convert back (histretch/README.md:4) */
  UWIP_ORDER_LITERAL = 1   /* as written: back-conversion before merge => colour-space round trip  */
} uwip_order;

typedef struct uwip_ctx uwip_ctx;

/* ---- context ------------------------------------------------------------------------------ */
int uwip_version(void);
/* replaces cuda::setDevice(0) + implicit OpenCV state (histretch.cpp:121-141). */
int uwip_create(int device, uwip_ctx** out);
void uwip_destroy(uwip_ctx* ctx);
/* last error text of this context (ctx may be NULL: error of the last failed uwip_create). */
const char* uwip_last_error(const uwip_ctx* ctx);
/* use an existing cudaStream_t (e.g. torch's current stream) instead of the context's own. */
int uwip_set_stream(uwip_ctx* ctx, void* cuda_stream);
int uwip_synchronize(uwip_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches). */
int64_t uwip_launch_count(const uwip_ctx* ctx);
/* device time in ms of the kernels whose name contains `tag`, accumulated since the last reset
 * when profiling is enabled with uwip_profile(ctx, 1); used for bench.py's roofline object. */
int uwip_profile(uwip_ctx* ctx, int enable);
int uwip_profile_read(uwip_ctx* ctx, const char* tag, double* total_ms, int64_t* launches);

/* staging helpers for host languages without a CUDA binding */
int uwip_device_alloc(uwip_ctx* ctx, size_t bytes, void** dptr);
int uwip_device_free(uwip_ctx* ctx, void* dptr);
int uwip_host_alloc(uwip_ctx* ctx, size_t bytes, void** hptr); /* pinned */
int uwip_host_free(uwip_ctx* ctx, void* hptr);
int uwip_copy_h2d(uwip_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes); /* async */
int uwip_copy_d2h(uwip_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes); /* async */

/* ---- modules/common/preprocessing.{h,cpp} --------------------------------------------------- */
/* int numChannel(char)  preprocessing.h:112, preprocessing.cpp:147-152 */
int uwip_num_channel(char c);
/* int numSpace(char)    preprocessing.h:115, preprocessing.cpp:154-161 */
int uwip_num_space(char c);
/* void getHistogram(cv::Mat*, cv::Mat*)  preprocessing.h:38, preprocessing.cpp:25-34:
 * 256-bin count of an 8U plane, delivered as float32[256] like calcHist's CV_32F column. */
int uwip_histogram_u8(uwip_ctx* ctx, const uint8_t* plane, int width, int height, size_t pitch,
                      float hist[256]);
int uwip_histogram_u8_dev(uwip_ctx* ctx, const uint8_t* d_plane, int width, int height,
                          float* d_hist);
/* void imgChannelStretch(cv::Mat, cv::Mat, int lo=0, int hi=100)  preprocessing.h:66,
 * preprocessing.cpp:74-105 (and imgChannelStretchGPU :109-144).  src == dst (in place) is what
 * every reference caller does.  Requires 0 <= lo < hi <= 100.  Optional out-params receive the
 * percentile bins (low may be -1 when lo == 0). */
int uwip_channel_stretch_u8(uwip_ctx* ctx, const uint8_t* src, size_t src_pitch, uint8_t* dst,
                            size_t dst_pitch, int width, int height, int lo, int hi, int* low_bin,
                            int* high_bin);
int uwip_channel_stretch_u8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int width,
                                int height, int lo, int hi);
/* the same for PITCHED device planes - what cv::cuda::GpuMat holds (cudaMallocPitch), i.e. the arguments of
 * imgChannelStretchGPU (preprocessing.cpp:109-144); stream ordered, does not synchronise */
int uwip_channel_stretch_u8_dev_pitched(uwip_ctx* ctx, const uint8_t* d_src, size_t src_pitch,
                                        uint8_t* d_dst, size_t dst_pitch, int width, int height, int lo,
                                        int hi);

/* ---- modules/histretch/src/histretch.cpp:219-254 (the -c=<letters> channel loop) ------------ */
/* channels: ordered letters; every letter of the CLI is built - RGB, HSV, HLS ('hsl'), Lab ('Lab') and
 * YCrCb ('YCX'), each equal to cv2 4.13.0 on all 2^24 triples (SURVEY 8f row N2); unknown letters are skipped like the CLI does.
 * The CLI hard-codes lo=2, hi=98 (histretch.cpp:154). */
int uwip_histretch_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t src_pitch, uint8_t* dst,
                        size_t dst_pitch, int width, int height, const char* channels, int lo,
                        int hi, int order, int hsv_round);
int uwip_histretch_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_frames,
                            int width, int height, const char* channels, int lo, int hi, int order,
                            int hsv_round);

/* ---- modules/aclahe ------------------------------------------------------------------------ */
/* cv::CLAHE::apply as called at aclahe.cpp:175-187, functions.py:24-27, aclahe/python/main.py:19-20
 * (8-bit plane; clip <= 0 disables clipping). */
int uwip_clahe_u8(uwip_ctx* ctx, const uint8_t* src, size_t src_pitch, uint8_t* dst,
                  size_t dst_pitch, int width, int height, double clip, int tiles_x, int tiles_y);
int uwip_clahe_u8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_planes, int width,
                      int height, double clip, int tiles_x, int tiles_y);
/* float aclaheEntropy(cv::Mat) aclahe.cpp:58,228-248 (flavour 0) / Entropia functions.py:14-19
 * (flavour 1, float32 throughout). */
int uwip_entropy_u8(uwip_ctx* ctx, const uint8_t* plane, int width, int height, size_t pitch,
                    int flavour, float* entropy);
/* cv2.GaussianBlur(img,(3,3),0) pre-filter, ACLAHE.py:15 */
int uwip_gaussian_blur3_u8(uwip_ctx* ctx, const uint8_t* src, size_t src_pitch, uint8_t* dst,
                           size_t dst_pitch, int width, int height);
/* the sweep of aclahe.cpp:180-193 / ACLAHE.py:38-47 for ONE grid size: entropies of
 * CLAHE(plane, clip_i, tiles) for n_clips clip limits, without writing the images (SURVEY 8f N1). */
int uwip_clahe_entropy_sweep_u8(uwip_ctx* ctx, const uint8_t* plane, int width, int height,
                                size_t pitch, int tiles, const double* clips, int n_clips,
                                int flavour, float* entropies);
/* the whole sweep of aclahe.cpp:160-193 / ACLAHE.py:20-47 in one call: n_frames device planes x n_grids square grids
 * (the reference's 2, 4, 8, 16, 32) x n_clips clip limits -> entropies [n_frames][n_grids][n_clips] (HOST pointer, for a
 * host-side knee search; uwip_aclahe_params_u8_dev does the whole parameter search on the device).  Synchronises the stream. */
int uwip_clahe_entropy_sweep_u8_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n_frames, int width, int height,
                                    const int* grids, int n_grids, const double* clips, int n_clips,
                                    int flavour, float* entropies);
/* frame wrapper aclahe.cpp:152-154 + the stubbed tail :214-218: BGR->HSV, CLAHE on V, HSV->BGR */
int uwip_aclahe_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t src_pitch, uint8_t* dst,
                     size_t dst_pitch, int width, int height, double clip, int tiles_x,
                     int tiles_y, int hsv_round);
int uwip_aclahe_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_frames,
                         int width, int height, double clip, int tiles_x, int tiles_y,
                         int hsv_round);

/* ---- automatic CLAHE parameters: ParametrosACLAHE (ACLAHE.py:9-129) on the device ------------------------------------ */
/* loop: which sweep of ACLAHE.py:38-47 to run.  REPAIRED evaluates all 50 clip limits per block size (what the code
 * intends); AS_COMMITTED is the file as it stands (the sweep body lost its indentation, the curves are all zero and the clip
 * limit degenerates to 0: crowd.png -> (8, 0)). */
typedef enum uwip_aclahe_loop {
  UWIP_ACLAHE_LOOP_REPAIRED = 0,
  UWIP_ACLAHE_LOOP_AS_COMMITTED = 1
} uwip_aclahe_loop;
/* For each of n equal-size device planes: GaussianBlur 3x3 -> entropy of CLAHE(blurred, k, c) for k in 2, 4, 8, 16, 32 and
 * c in 0, 0.5 .. 24.5 -> per block size the knee of the entropy curve (scipy's curve_fit double exponential restated as
 * MINPACK lmdif, not-a-knot spline, curvature argmax; csrc/aclahe_knee.h) -> CL = max of the five knees (an integer 0..48,
 * used directly as the clip limit) -> BS = the block size whose entropy of CLAHE(blurred, BS, CL), rounded to float16, is
 * the last maximum.  d_bs, d_cl: device int32[n].  A plane whose fit fails (the reference raises RuntimeError) gets
 * BS = CL = -1 and the frame flag UWIP_FRAME_ACLAHE_NOFIT.  Planes too small for a 32 x 32 grid are refused
 * (UWIP_ERR_INVALID).  Stream ordered, does not synchronise. */
int uwip_aclahe_params_u8_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n_planes, int width, int height, int loop,
                              int32_t* d_bs, int32_t* d_cl);
/* automatic aclahe on n device frames: V of each frame -> uwip_aclahe_params_u8_dev -> BGR->HSV, CLAHE on V with the
 * frame's own (BS, CL), HSV->BGR.  clip and tiles_x x tiles_y are used only for frames whose fit failed.  d_bs, d_cl:
 * optional device int32[n] outputs (NULL: not returned).  Stream ordered, does not synchronise. */
int uwip_aclahe_bgr8_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_frames, int width, int height,
                              int loop, int hsv_round, double clip, int tiles_x, int tiles_y, int32_t* d_bs,
                              int32_t* d_cl);
/* automatic CLAHE on n device u8 planes, the grey prototype (modules/aclahe/python/main.py:18-20) for a batch: the plane's
 * (BS, CL) from uwip_aclahe_params_u8_dev (which blurs internally, ACLAHE.py:15), then createCLAHE(CL, (BS, BS)).apply of the
 * unblurred plane.  A plane whose fit failed gets BS = CL = -1, UWIP_FRAME_ACLAHE_NOFIT, and CLAHE with clip and
 * tiles_x x tiles_y.  d_src may equal d_dst.  d_bs, d_cl: optional device int32[n] outputs (NULL: not returned).  The size
 * refusals are those of uwip_aclahe_params_u8_dev.  A plane's bytes do not depend on the batch it is in.  Stream ordered,
 * does not synchronise. */
int uwip_aclahe_u8_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_planes, int width, int height,
                            int loop, double clip, int tiles_x, int tiles_y, int32_t* d_bs, int32_t* d_cl);

/* ---- modules/bgdehaze ---------------------------------------------------------------------- */
typedef struct uwip_dehaze_params {
  int window;  /* dark-channel window of Background_light; default 15 (main.py:28).  The transmission
                  window is ALWAYS 15 because dehazed_BG calls refined_t without w (BGDehaze.py:52) */
  int radius;  /* guided filter radius, 40 (BGDehaze.py:41,72); 1..128: the window sums of the guide
                  moments are 32-bit, exact while (2r+1)^2 255^2 < 2^32 */
  double eps;  /* guided filter eps, 1e-3 (BGDehaze.py:42,73); >= 1e-3: the coefficients are stored in
                  fixed point whose step grows as eps shrinks */
  double tmin; /* transmission floor, 0.2 (BGDehaze.py:40)      */
} uwip_dehaze_params;
void uwip_dehaze_defaults(uwip_dehaze_params* p);

/* boxfilter(I, r)  guidedfilter.py:23-51: (2r+1)^2 window SUM of a float64 plane, windows truncated at the borders
 * (what cv2.boxFilter(normalize=False, BORDER_CONSTANT) computes).  Stage entry for parity; direct sums. */
int uwip_boxfilter_f64(uwip_ctx* ctx, const double* src, int width, int height, int r, double* dst);
/* guided_filter(I, p, r, eps)  guidedfilter.py:54-103 for a guide of the form I = guide8 / range, guide8 an 8-bit
 * three-channel image (every guide on the path is one: normI of main.py:17, normYiCrCb of BGDehaze.py:77-80);
 * p float64 in [0, 1.6] (held on a 2^-28 grid), q float64, r 1..128, eps >= 1e-3.  Runs the same two marches as the chain's filters. */
int uwip_guided_filter_u8(uwip_ctx* ctx, const uint8_t* guide, size_t pitch, int width, int height,
                          int range, const double* p, int r, double eps, double* q);
/* Background_light(normI, w)  BGDehaze.py:14-26 on the frame normalised as main.py:17.
 * Tie rule: first flat index of the minimum (SURVEY 8a-D1).  B in B,G,R order. */
int uwip_background_light_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int width,
                               int height, int window, double B[3], int64_t idx[2]);
/* transmission_map(normI, w)  BGDehaze.py:28-37: planes t_blue, t_green (float64, width*height) */
int uwip_transmission_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int width, int height,
                           int window, double* t_blue, double* t_green);
/* refined_t(normI)  BGDehaze.py:39-48 (guided_filter of guidedfilter.py:54-103 on max(t,tmin)) */
int uwip_refined_transmission_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int width,
                                   int height, const uwip_dehaze_params* p, double* t_blue,
                                   double* t_green);
/* RC_correction(normI, w)  BGDehaze.py:59-69: restored, float64 H x W x 3 (B,G,R interleaved) */
int uwip_rc_correction_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int width, int height,
                            const uwip_dehaze_params* p, double* restored);
/* generate_results(src, dest, adaptiveExp_map)  bgdehaze/main.py:14-20 minus file I/O:
 * dst8 = sat(rint(out*255)) (what imwrite hands to the encoder); out_f64 (optional, may be NULL)
 * = adaptiveExp_map(normI, w)  BGDehaze.py:71-89, float64 H x W x 3. */
/* adaptiveExp_map(normI, w)  BGDehaze.py:71-89, stage by stage (a test hook: one frame, not on the throughput path).  One
 * full run of uwip_bgdehaze_bgr8, then its intermediates, width*height each, row-major:
 * ycc = Yi | Cri << 8 | Cbi << 16 | Yj << 24 (YCrCb of (normI*255).astype(uint8) and luma of (restored*255).astype(uint8),
 * BGDehaze.py:75-78); splane = rint(S 2^28) of the exposure ratio S (BGDehaze.py:83; 0 where S is 0/0); refined_s = the
 * refined S (BGDehaze.py:85, float32); restored = RC_correction's output and out = adaptiveExp_map's (float64 H x W x 3,
 * out NaN for a flagged frame); stats = yi_min, yi_max, yj_min, yj_max (joint three-channel extremes of the two YCrCb
 * images) and the frame's NaN flag word (nonzero: UWIP_FRAME_NAN). */
int uwip_exposure_stages_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int width, int height,
                              const uwip_dehaze_params* p, uint32_t* ycc, uint32_t* splane, float* refined_s,
                              double* restored, double* out, uint32_t stats[5]);
int uwip_bgdehaze_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t src_pitch, uint8_t* dst8,
                       size_t dst_pitch, int width, int height, const uwip_dehaze_params* p,
                       double* out_f64);
int uwip_bgdehaze_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_frames,
                           int width, int height, const uwip_dehaze_params* p);

/* ---- the chain: histretch -c=<channels> | aclahe | bgdehaze on a batch of frames ------------- */
typedef struct uwip_chain_params {
  char channels[16];  /* histretch letters, default "V"            */
  int lo, hi;         /* percentiles, default 1 / 99 (BASELINE config 1; the CLI default is 2 / 98) */
  int order;          /* uwip_order                                 */
  int hsv_round;      /* uwip_hsv_round                             */
  double clip;        /* CLAHE clip limit, default 2.0              */
  int tiles_x, tiles_y; /* CLAHE grid, default 8 x 8                */
  uwip_dehaze_params dehaze;
} uwip_chain_params;
void uwip_chain_defaults(uwip_chain_params* p);

/* device resident: n_frames contiguous bgr8 frames in, same out (d_src may equal d_dst). */
int uwip_chain_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_frames,
                        int width, int height, const uwip_chain_params* p);
/* the chain with automatic CLAHE parameters: the parameters of each frame are found on the V plane of the frame that
 * enters CLAHE (the histretch output, as the aclahe CLI does with its input); p->clip and p->tiles_* apply only to frames
 * whose fit failed (UWIP_FRAME_ACLAHE_NOFIT).  d_bs, d_cl: optional device int32[n] outputs (NULL: not returned).  A frame's
 * bytes do not depend on the batch it is in. */
int uwip_chain_bgr8_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_frames, int width, int height,
                             const uwip_chain_params* p, int loop, int32_t* d_bs, int32_t* d_cl);
/* host buffers (pinned memory recommended): H2D, chain, D2H pipelined over sub-batches through two staging buffers per
 * direction; the sub-batch sizes ramp up and down in whole CTA waves (csrc/e2e_schedule.h) so that only a few frames'
 * upload and download are exposed.  The bytes are those of the device-resident call whatever the schedule.  Returns after
 * the last download has completed. */
int uwip_chain_bgr8(uwip_ctx* ctx, const uint8_t* src, uint8_t* dst, int n_frames, int width,
                    int height, const uwip_chain_params* p);

/* per-frame status bits of the LAST uwip_chain_bgr8[_auto][_dev] / uwip_bgdehaze_bgr8_dev / uwip_aclahe_params_u8_dev /
 * uwip_aclahe_bgr8_auto_dev / uwip_aclahe_u8_auto_dev / uwip_jpeg_decode_{bgr8,u8}_batch[_oriented] / uwip_jpeg_decode_batch_ex call on
 * this context (synchronises the stream).  UWIP_FRAME_NAN: the reference's
 * adaptiveExp_map is NaN for the whole frame (S = 0/0 where Yi = Yj = 0, BGDehaze.py:83, spreads through the box filters
 * and the final min-max; SURVEY 8a-D9) - the 8-bit output is then all zeros, exactly what imwrite would store.
 * UWIP_FRAME_ACLAHE_NOFIT: an automatic-CLAHE call could not fit an entropy curve of the frame (the reference's curve_fit
 * raises RuntimeError); the frame's BS = CL = -1 and it was processed with the fixed clip limit and grid.
 * UWIP_FRAME_JPEG_BAD (set by the batched JPEG readers): the file's entropy-coded data is bad - an invalid Huffman code, a
 * coefficient past 63, the data ending before the last block or the wrong number of restart markers; the frame is all zeros
 * (libjpeg's recovery from corrupt data is not restated). */
#define UWIP_FRAME_NAN 1
#define UWIP_FRAME_ACLAHE_NOFIT 2
#define UWIP_FRAME_JPEG_BAD 4
int uwip_last_frame_flags(uwip_ctx* ctx, int n_frames, int32_t* flags_host);

/* ---- modules/videostrip: calcBlur (SURVEY 8f row N4, the frame-quality gate in front of the chain) */
/* float calcBlur(Mat frame), videostrip.cpp:170-184 (declared videostrip.hpp:98; calcBlurGPU :39-60 is the
 * cv::cuda twin): BGR2GRAY -> Laplacian(grey, laplacian, grey.type(), CV_16S) = 8-bit output, aperture 3
 * (kernel [2 0 2; 0 -8 0; 2 0 2], reflect-101) -> meanStdDev -> (float)stdev.  aperture = 3 is that call;
 * aperture = 1 is the kernel [0 1 0; 1 -4 1; 0 1 0] that calcBlurGPU requests (videostrip.cpp:48).
 * mean_std (optional): the doubles meanStdDev returns, {mean, stdev}.  lap (optional): the 8-bit Laplacian. */
int uwip_calc_blur_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int width, int height,
                        int aperture, float* stdev, double* mean_std, uint8_t* lap, size_t lap_pitch);
/* batch on device memory: d_mean_std[2f], d_mean_std[2f+1] = mean, stdev of frame f (stream-ordered) */
int uwip_calc_blur_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, int n_frames, int width, int height,
                            int aperture, double* d_mean_std);

/* ---- JPEG files to and from the device (SURVEY 8f row N3) ------------------------------------ */
/* imread / imwrite around the chain (histretch.cpp:158,268, aclahe.cpp:135, bgdehaze/main.py:16,19) for baseline JPEG
 * files: nvJPEG decodes into the bgr8 device layout the chain reads and encodes from the one it writes, so a frame crosses
 * PCIe as its compressed bytes only.  The decoded pixels are nvJPEG's (its IDCT is not bit-identical to libjpeg-turbo's:
 * a few levels from cv2.imread, mostly the 4:2:0 chroma upsampling: max 4, mean 0.6 on the test frame); encoding is 4:2:0 at `quality` (cv2.imwrite's default is 95). */
int uwip_jpeg_info(uwip_ctx* ctx, const uint8_t* jpeg, size_t len, int* width, int* height);
int uwip_jpeg_decode_bgr8_dev(uwip_ctx* ctx, const uint8_t* jpeg, size_t len, uint8_t* d_bgr, int width,
                              int height);
/* out == NULL: only *out_len (the size of the stream) is returned */
int uwip_jpeg_encode_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_bgr, int width, int height, int quality,
                              uint8_t* out, size_t cap, size_t* out_len);
/* JPEG in -> histretch -> aclahe -> bgdehaze on the device -> JPEG out */
int uwip_chain_jpeg(uwip_ctx* ctx, const uint8_t* jpeg_in, size_t len_in, const uwip_chain_params* p,
                    int quality, uint8_t* jpeg_out, size_t cap, size_t* len_out);
/* Batched encoder whose files are byte-identical to cv2.imwrite / cv2.imencode(".jpg", frame, [IMWRITE_JPEG_QUALITY, quality])
 * with libjpeg-turbo: baseline JFIF, 4:2:0, the standard quantisation tables scaled by quality and the standard Huffman tables;
 * no restart markers, no optimised Huffman tables, not progressive (csrc/jpegenc.h restates the arithmetic).  This is the
 * writer of the reference's command lines (histretch.cpp:268, bgdehaze/main.py:19), so device output can be compared with
 * reference files byte for byte; the nvJPEG entry points above write other bytes.
 * uwip_jpeg_encode_bound: the largest file a width x height frame can produce (every coefficient coded with the longest code,
 * every scan byte stuffed), 0 for sizes outside 1..65535.  libjpeg itself refuses sizes above 65500. */
size_t uwip_jpeg_encode_bound(int width, int height);
/* n_frames contiguous bgr8 device frames -> frame f's file at d_out + f * out_stride (device memory, out_stride >=
 * uwip_jpeg_encode_bound(width, height); the slot is also the encoder's scratch) and its length in d_len[f] (device
 * uint64).  Refuses out_stride below the bound, quality outside 1..100 and sizes outside 1..65535 (UWIP_ERR_INVALID).
 * A frame's bytes do not depend on the batch it is in.  Stream ordered, does not synchronise. */
int uwip_jpeg_encode_bgr8_batch_dev(uwip_ctx* ctx, const uint8_t* d_bgr, int n_frames, int width, int height, int quality,
                                    uint8_t* d_out, size_t out_stride, uint64_t* d_len);
/* The grey twin: the bytes of cv2.imwrite / cv2.imencode(".jpg", plane, [IMWRITE_JPEG_QUALITY, quality]) for a 2-D u8 plane -
 * one component (h = v = 1, quantisation table 0, Huffman tables 0), an MCU of one block, the right and bottom edges
 * replicated into the last blocks, JFIF APP0.  Same slot layout, refusals and guarantees as the bgr8 call, with
 * uwip_jpeg_encode_u8_bound in place of uwip_jpeg_encode_bound. */
size_t uwip_jpeg_encode_u8_bound(int width, int height);
int uwip_jpeg_encode_u8_batch_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n_frames, int width, int height, int quality,
                                  uint8_t* d_out, size_t out_stride, uint64_t* d_len);

/* Batched decoder whose pixels equal cv2.imread / cv2.imdecode(file, IMREAD_COLOR) with libjpeg-turbo (islow IDCT, fancy
 * upsampling, csrc/jpegdec.h restates the arithmetic), the reader of the reference's command lines (histretch.cpp:158,
 * bgdehaze/main.py:16), so that a .jpg input gives the device chain the reference's pixels; uwip_jpeg_decode_bgr8_dev above
 * gives nvJPEG's.  Accepted: baseline and extended sequential Huffman, 8-bit, one scan, grey or YCbCr 4:4:4, 4:2:2, 4:4:0,
 * 4:2:0, any restart interval, any tables.  The pixels are the stored orientation (cv2.IMREAD_COLOR |
 * IMREAD_IGNORE_ORIENTATION), which is what cv2.imdecode(file, IMREAD_COLOR) returns for every file without an Exif
 * orientation; uwip_jpeg_decode_bgr8_batch_oriented below applies it.
 * n host JPEG files (jpegs[f], lens[f]) of one size -> the bgr8 frames cv2.imdecode(file, IMREAD_COLOR) returns, contiguous
 * at d_bgr.  Tables, sampling and restart interval may differ per file; width x height may not (UWIP_ERR_INVALID).
 * Unsupported coding: UWIP_ERR_UNSUPPORTED.  Bad entropy-coded data: the frame is zeros and UWIP_FRAME_JPEG_BAD is set
 * (uwip_last_frame_flags).  The headers are parsed and the files copied to pinned staging before the call returns, so the
 * caller's memory is free again then.  A frame's pixels do not depend on the batch it is in.  Stream ordered, does not
 * synchronise.  n_frames <= 65535. */
int uwip_jpeg_decode_bgr8_batch(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames,
                                uint8_t* d_bgr, int width, int height);
/* The grey twin: the u8 planes cv2.imdecode(file, IMREAD_GRAYSCALE) returns, contiguous at d_planes.  For a grey file these
 * are its samples; for a YCbCr file its Y component (islow and range limit, cropped; the chroma is entropy-decoded but not
 * transformed), which is not cvtColor(BGR2GRAY) of the colour pixels.  Accepts, refuses and flags exactly as
 * uwip_jpeg_decode_bgr8_batch. */
int uwip_jpeg_decode_u8_batch(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames,
                              uint8_t* d_planes, int width, int height);
/* The readers above with each file's Exif orientation applied as cv2.imdecode(file, IMREAD_COLOR) and
 * cv2.imdecode(file, IMREAD_GRAYSCALE) apply it with their default flags: flipped for orientations 2, 3, 4, transposed for
 * 5 to 8 (uwip_jpeg_orientation gives the value).  width x height is the size after orientation: a file's stored size must
 * be width x height for orientations 1 to 4 and height x width for 5 to 8 (UWIP_ERR_INVALID otherwise), so a batch may mix
 * orientations.  They accept, refuse and flag exactly as the readers above; a flagged frame is zeros of width x height. */
int uwip_jpeg_decode_bgr8_batch_oriented(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames,
                                         uint8_t* d_bgr, int width, int height);
int uwip_jpeg_decode_u8_batch_oriented(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames,
                                       uint8_t* d_planes, int width, int height);
/* The Exif orientation, 1 to 8, that cv2.imdecode (cv2 4.13.0) applies to a file: the first Exif APP1 before the scan whose
 * IFD0 holds an orientation tag decides, and 1 stands for no tag or a value outside 1..8.  Runs the host marker reader of
 * the readers above: UWIP_ERR_INVALID / UWIP_ERR_UNSUPPORTED for a header they refuse.  No context, no device. */
int uwip_jpeg_orientation(const uint8_t* jpeg, size_t len, int* orientation);
/* The exact reader for sequential and progressive files alike, in one call: everything the four readers above accept,
 * plus progressive Huffman files (SOF2) of the same samplings, such as cv2.imwrite(.., [IMWRITE_JPEG_PROGRESSIVE, 1]) and
 * Pillow's save(.., progressive=True) write.  flags: UWIP_JPEG_GREY for the planes of cv2.imdecode(file, IMREAD_GRAYSCALE)
 * in place of bgr8 frames, UWIP_JPEG_ORIENT for the Exif orientation applied (width x height then the size after it), as
 * the readers above.  A batch may mix sequential and progressive files; a frame's pixels do not depend on the batch it is
 * in.  Every scan is entropy-decoded, in grey output too.  Refused as the readers above (UWIP_ERR_INVALID,
 * UWIP_ERR_UNSUPPORTED), and besides: bad Ss / Se / Ah / Al in a progressive scan (UWIP_ERR_INVALID); a scan whose Ah is
 * not the Al of the previous scan of the same coefficients, an AC scan before the component's DC scan, more than 128 scans,
 * and a progression that is incomplete at EOI - some coefficient of some component not refined down to Al = 0
 * (UWIP_ERR_UNSUPPORTED: libjpeg-turbo decodes such files with block smoothing, which this reader does not restate).  Bad
 * entropy-coded data zeroes the frame and sets UWIP_FRAME_JPEG_BAD as above, and so does a progressive file whose data ends
 * inside a scan.  The headers are parsed and the files copied to pinned staging before the call returns.  Stream ordered,
 * does not synchronise.  n_frames <= 65535. */
#define UWIP_JPEG_GREY 1
#define UWIP_JPEG_ORIENT 2
int uwip_jpeg_decode_batch_ex(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames,
                              uint8_t* d_out, int width, int height, int flags);
/* The marker reader of uwip_jpeg_decode_batch_ex over a whole file, without a context or a device: the size of the image
 * cv2.imdecode returns (after the Exif orientation: width and height swapped for orientations 5 to 8), the orientation
 * (1 to 8) and whether the file is progressive.  Returns what uwip_jpeg_decode_batch_ex would refuse the file with, or
 * UWIP_OK (also for a file whose entropy-coded data is bad: that is found by decoding). */
int uwip_jpeg_probe(const uint8_t* jpeg, size_t len, int* width, int* height, int* orientation, int* progressive);
/* per-frame statistics of the last batched JPEG decode (either reader; synchronises): stats[2f] = subsequence decodes the
 * in-CTA synchronisation repeated, stats[2f + 1] = subsequences the cross-CTA fix-up re-decoded. */
int uwip_jpeg_decode_stats(uwip_ctx* ctx, int n_frames, int32_t* stats);

/* ---- synthetic input + checksums (SURVEY 8d) ------------------------------------------------- */
/* frames first_frame .. first_frame+n_frames-1 of the integer-only generator (twin of
 * oracle/uwip_oracle.py:synth_frame) written to device memory. */
int uwip_synth_bgr8_dev(uwip_ctx* ctx, uint8_t* d_dst, uint32_t seed, int first_frame, int n_frames,
                        int width, int height);
/* per-frame 64-bit position-weighted checksum of device frames (for shard-vs-single-GPU equality) */
int uwip_checksum_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, int n_frames, int width, int height,
                           uint64_t* sums_host);

#ifdef __cplusplus
}
#endif
#endif /* UWIP_H */
