/*
 * trs_b200.h — C ABI of the B200-native batched observation path for Triton-Racer-Sim.
 *
 * The reference (pure Python) has no FFI of its own: its boundary for this path is the
 * `Component` plugin API (TritonRacerSim/components/component.py:3-28).  The Python mirror of
 * that API lives in triton-racer-sim_b200/components.py and reaches the sm_100a kernels only
 * through the entry points declared here (ctypes, see INTEGRATION.md).  Every entry point names
 * the reference code it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary
 *   - every function returns int: 0 = ok, >0 = cudaError_t, <0 = TRS_E_* argument error;
 *     trs_last_error() returns a thread-local message for the last non-zero return
 *   - "_dev" pointers are device pointers (contiguous); frame pointers should be 16-byte aligned
 *   - work is enqueued on the caller's stream (a cudaStream_t passed as void*) and the call
 *     returns without synchronising; the *_host entry points synchronise before returning
 *   - frames are (N,H,W,3) uint8 RGB, HWC interleaved: the input contract of
 *     TritonRacerSim/components/gyminterface.py:95-104
 */
#ifndef TRS_B200_H
#define TRS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRS_VERSION 100

#define TRS_E_ARG      (-1)  /* null pointer / bad size / bad enum                */
#define TRS_E_STATE    (-2)  /* e.g. locate before set_track                       */
#define TRS_E_RANGE    (-3)  /* frame too large for the on-chip working set        */
#define TRS_E_NODEVICE (-4)  /* no sm_100 device                                   */

#define TRS_MAX_HSV 4        /* colour ranges accepted (only the last writer of each channel matters) */

typedef struct trs_ctx trs_ctx;

/* Parameters of ImgPreprocessing — names follow core/config.py:15-28 (preprocessing_*). */
typedef struct trs_preproc_params {
    double contrast_ratio;        /* preprocessing_contrast_enhancement_ratio   (config.py:18) */
    double contrast_offset;       /* preprocessing_contrast_enhancement_offset  (config.py:19) */
    double brightness_baseline;   /* preprocessing_brightness_baseline          (config.py:21) */
    int32_t dynamic_brightness;   /* preprocessing_dynamic_brightness_enabled   (config.py:20) */
    int32_t color_filter_enabled; /* preprocessing_color_filter_enabled         (config.py:22) */
    int32_t n_hsv;                /* len(preprocessing_color_filter_hsvs)       (config.py:23) */
    int32_t edge_enabled;         /* preprocessing_edge_detection_enabled       (config.py:25) */
    double hsv_lo[TRS_MAX_HSV][3];/* lower (H,S,V) bound of each range; rounded to int32 half-to-even (out of range -> INT_MIN) before the compare, as cv2.inRange does */
    double hsv_hi[TRS_MAX_HSV][3];/* upper (H,S,V) bound, inclusive, same rounding */
    int32_t color_dest[TRS_MAX_HSV]; /* preprocessing_color_filter_destination_channels (config.py:24) */
    int32_t edge_dest;            /* preprocessing_edge_detection_destination_channel (config.py:28) */
    double canny_a;               /* preprocessing_edge_detection_threshold_a   (config.py:26) */
    double canny_b;               /* preprocessing_edge_detection_threshold_b   (config.py:27) */
} trs_preproc_params;

/* Parameters of the pilots' speed-control tail — core/config.py:65-66,76-80. */
typedef struct trs_spd_params {
    double threshold;             /* spd_ctl_threshold            */
    double reverse_multiplier;    /* spd_ctl_reverse_multiplier   */
    double break_multiplier;      /* spd_ctl_break_multiplier     */
    int32_t use_break;            /* spd_ctl_break                */
    int32_t smooth_steering;      /* smooth_steering_enabled      */
    double smooth_threshold;      /* smooth_steering_threshold    */
    int32_t numpy_legacy_promotion; /* 0: NumPy >= 2 scalar promotion (NEP 50): np.float32 model output * 20, * threshold and the speed gap stay
                                     *    float32 (what the reference computes under the numpy this image pins);
                                     * 1: NumPy 1.x promotion: the same expressions are float64 (the TF2-era stacks the reference was written for) */
    int32_t reserved;
} trs_spd_params;

/* Per-call statistics written by trs_preprocess (all counters are sums over the N frames). */
enum {
    TRS_STAT_FRAMES = 0,     /* frames processed                                   */
    TRS_STAT_MASK0 = 1,      /* set pixels of colour range 0..3                    */
    TRS_STAT_MASK1 = 2,
    TRS_STAT_MASK2 = 3,
    TRS_STAT_MASK3 = 4,
    TRS_STAT_EDGE = 5,       /* Canny edge pixels after hysteresis                 */
    TRS_STAT_STRONG = 6,     /* pixels above the high threshold after NMS          */
    TRS_STAT_CAND = 7,       /* NMS survivors above the low threshold              */
    TRS_STAT_HYST_SWEEPS = 8,/* hysteresis sweeps summed over frames               */
    TRS_STAT_ROI_SUM = 9,    /* sum of all ROI bytes (brightness statistic)        */
    /* cycle accounting of thread 0 of every CTA (SM clocks, summed over CTAs) — only in builds with -DTRS_PHASE_TIMERS
       (tools/phase_timing.py); the meaning of slots 12..14 depends on the kernel (see preproc_fast.cuh) */
    TRS_STAT_T_WAIT_FRAME = 10,       /* waiting for the TMA frame load                         */
    TRS_STAT_T_STRIP_WALK = 11,       /* P1: Sobel strip walk + colour masks                    */
    TRS_STAT_T_PHASE_A = 12,          /* resident kernel: NMS           | store-warp kernel: waiting for the store warps */
    TRS_STAT_T_PHASE_B = 13,          /* resident kernel: hysteresis    | store-warp kernel: NMS                         */
    TRS_STAT_T_PHASE_C = 14,          /* resident kernel: output        | store-warp kernel: hysteresis                  */
    TRS_STAT_T_TOTAL = 15,            /* whole frame loop                                        */
    TRS_STAT_COUNT = 24
};

int trs_version(void);
const char* trs_last_error(void);
/* Number of kernels this library has launched in this process (all contexts); bench.py reports it. */
unsigned long long trs_kernel_launches(void);

/* One context per GPU.  Holds the uploaded parameter tables and the waypoint table. */
int trs_ctx_create(int device, trs_ctx** out);
int trs_ctx_destroy(trs_ctx* ctx);
/* Properties of the device the context is bound to (SM count, opt-in shared memory per block). */
int trs_ctx_device_info(trs_ctx* ctx, int* sm_count, int* smem_optin_bytes, int* cc_major, int* cc_minor);

/* Replaces reading self.cfg[...] inside ImgPreprocessing (img_preprocessing.py:41-50,66-68,77-78,84-86). */
int trs_set_preproc_params(trs_ctx* ctx, const trs_preproc_params* p);

/*
 * Replaces ImgPreprocessing.__process (img_preprocessing.py:37-54) for N frames, fused with the
 * pilot's float normalisation (keras_pilot.py:49-50) when out_f32_dev is given.
 *   in_dev      (N,H,W,3) u8
 *   out_u8_dev  (N,H,W,3) u8  `cam/processed_img`            — nullable
 *   out_f32_dev (N,H,W,3) f32 `processed_img / 255`          — nullable
 *   stats_dev   TRS_STAT_COUNT x u64, accumulated atomically  — nullable
 */
int trs_preprocess(trs_ctx* ctx, const uint8_t* in_dev, int n, int h, int w,
                   uint8_t* out_u8_dev, float* out_f32_dev, unsigned long long* stats_dev,
                   void* stream);

/*
 * Replaces the camera resize (camera.py:36, nearest neighbour), a rows/cols window crop and the
 * float normalisation (keras_pilot.py:49-50, keras_train.py:41-42) for N frames.
 *   in_dev (N,h_in,w_in,3) u8; window rows [roi_y0,roi_y1) cols [roi_x0,roi_x1) of the source;
 *   the window is scaled to (h_out,w_out) with src = floor(dst*size_src/size_dst);
 *   out_f32_dev (N,h_out,w_out,3) f32 = u8/255 — nullable; out_u8_dev same shape u8 — nullable.
 */
int trs_normalise(trs_ctx* ctx, const uint8_t* in_dev, int n, int h_in, int w_in,
                  int roi_y0, int roi_y1, int roi_x0, int roi_x1, int h_out, int w_out,
                  float* out_f32_dev, uint8_t* out_u8_dev, void* stream);

/* Replaces LocationTracker.__init__ (track_data_process.py:69-75): upload the centre line (host pointer, n_wp x 3 f64). */
int trs_set_track(trs_ctx* ctx, const double* wp_xyz_host, int n_wp, double min_map, double max_map);

/*
 * Replaces LocationTracker.step/localize/__find_closest/__map (track_data_process.py:77-107) for N cars.
 *   xyz_dev (N,3) f64; idx_dev (N) i32 — nullable; segment_dev (N) f64 — nullable.
 *   Large batches keep a per-context scratch list (cars finished by a second kernel in the same stream): issue the
 *   calls of one context on one stream at a time, or use a context per stream.
 */
int trs_locate(trs_ctx* ctx, const double* xyz_dev, int n, int32_t* idx_dev, double* segment_dev,
               void* stream);

/*
 * Replaces the speed-control tail of KerasPilot.step (keras_pilot.py:80-95,99-118,142-153) and
 * calcThrottle/calcBreak (utils/mapping.py:23-35) for N cars.
 *   cur_spd_dev (N) f64 `gym/speed`; model_spd_dev (N) f32 = the model's speed output (before x20);
 *   model_steer_dev (N) f32 = the model's steering output;
 *   outputs (N) f64 each: `ai/steering`, `ai/throttle`, `ai/breaking`;
 *   spd_feature_dev (N) f32 = gym/speed / 20 (keras_pilot.py:68,100) — nullable.
 */
int trs_speed_control(trs_ctx* ctx, const double* cur_spd_dev, const float* model_spd_dev,
                      const float* model_steer_dev, int n, const trs_spd_params* p,
                      double* steering_dev, double* throttle_dev, double* breaking_dev,
                      float* spd_feature_dev, void* stream);

/*
 * Per-car control post-processing, the step after the speed controller (SURVEY.md 8(f)):
 *   ControlMultiplexer.step  TritonRacerSim/components/controlmultiplexer.py:24-43  usr/ai select by drive mode + AI launch locks (48-70)
 *   DriverAssistance.step    TritonRacerSim/components/driver_assistance.py:13-31    fused when speed_dev is given and assist_mode != 0
 *   mode_dev (n) int32: TRS_MODE_* (DriveMode.HUMAN / AI_STEERING / AI, components/controller.py:7-10)
 *   usr_dev, ai_dev, out_dev: (3, n) f64 = steering, throttle, breaking
 *   now_s: the clock (the reference's locks are ended by sleeping threads; here time is an argument)
 *   state, updated in place: last_mode_dev (n) int32, initially TRS_MODE_HUMAN; launch_times_dev (TRS_LAUNCH_SLOTS, n) f64,
 *   initially TRS_NEVER.  A lock is set at the latest launch and cleared at the earliest pending end time after it, as the
 *   reference's threads do; exact while at most TRS_LAUNCH_SLOTS lock threads would be pending at once.
 */
#define TRS_MODE_HUMAN 0
#define TRS_MODE_AI_STEERING 1
#define TRS_MODE_AI 2
#define TRS_LAUNCH_SLOTS 4
#define TRS_NEVER (-1.0e300)
typedef struct {
    int32_t throttle_lock_enabled;   /* ai_launch_boost_throttle_enabled  (core/config.py:57) */
    int32_t steering_lock_enabled;   /* ai_launch_lock_steering_enabled   (core/config.py:61) */
    int32_t assist_mode;             /* 0 off, 1 'steering', 2 'speed'    (drive_assist_limit_mode, core/config.py:105) */
    int32_t reserved;
    double throttle_lock_value;      /* ai_launch_boost_throttle_value    */
    double throttle_lock_duration;   /* ai_launch_boost_throttle_duration */
    double steering_lock_value;      /* ai_launch_lock_steering_value     */
    double steering_lock_duration;   /* ai_launch_lock_steering_duration  */
    double assist_k;                 /* drive_assist_limit_k              */
} trs_ctl_params;
int trs_control_mux(trs_ctx* ctx, const int32_t* mode_dev, const double* usr_dev, const double* ai_dev, const double* speed_dev,
                    int n, const trs_ctl_params* p, double now_s, int32_t* last_mode_dev, double* launch_times_dev,
                    double* out_dev, void* stream);
/* three_segment_map (TritonRacerSim/utils/mapping.py:9-16): [-1, 1] command -> PWM value around a neutral point. */
int trs_pwm_map(trs_ctx* ctx, const double* val_dev, int n, double min_map, double mid_map, double max_map, double* out_dev,
                void* stream);

/*
 * Tub ingestion (SURVEY.md 8(f) rank 1): batched decode of the records' JPEG files, replacing
 *   np.asarray(Image.open(img_path))      TritonRacerSim/components/keras_train.py:41,309
 * for the files the reference's recorder writes (Image.fromarray(img).save(path), components/datastorage.py:78: baseline, 8 bit,
 * YCbCr 4:2:0, one scan, no restart intervals).  Bit-exact with Pillow / libjpeg(-turbo) defaults (integer IDCT, fancy upsampling).
 *   blob_host     the N files back to back (pageable or pinned host memory)
 *   offsets_host  N + 1 byte offsets into blob_host (file k = [offsets[k], offsets[k+1]))
 *   out_u8_dev    (N, h, w, 3) uint8 RGB on the device; every file must be h x w
 * Parses on the host, uploads the files (about 5 KB per 120x160 record instead of 57.6 KB of pixels), decodes on the GPU;
 * synchronises `stream` before returning (the staging buffers are reused by the next call).
 * TRS_E_RANGE: a file is not a baseline 4:2:0 JPEG of the stated size (the message names the record).
 */
int trs_jpeg_decode_host(trs_ctx* ctx, const uint8_t* blob_host, const unsigned long long* offsets_host, int n, int h, int w,
                         uint8_t* out_u8_dev, void* stream);

/*
 * Gym telemetry ingestion (SURVEY.md 8(f) rank 2): the camera images of N simulator clients, replacing
 *   Image.open(BytesIO(base64.b64decode(json_packet["image"])))     TritonRacerSim/components/gyminterface.py:96-99
 * text_host holds the N base64 strings back to back (standard alphabet, '=' padding optional, white space ignored),
 * offsets_host N + 1 byte offsets into it.  The strings are decoded on the host (threads) and the JPEG files go through the same
 * path as trs_jpeg_decode_host.  TRS_E_RANGE: a string is not valid base64 or not a supported JPEG of the stated size.
 */
int trs_telemetry_decode_host(trs_ctx* ctx, const char* text_host, const unsigned long long* offsets_host, int n, int h, int w,
                              uint8_t* out_u8_dev, void* stream);

/*
 * Tub recording: batched JPEG encode of N device frames, replacing
 *   Image.fromarray(img).save(path)      TritonRacerSim/components/datastorage.py:78 (the recorder's cam/processed_img, manage.py:103-104)
 *   cv2.imwrite(path, img)               TritonRacerSim/utils/post_process.py (the same bytes at the same quality)
 * Baseline JPEG, YCbCr 4:2:0, libjpeg quality scaling, standard Huffman tables: byte-identical with Pillow / libjpeg(-turbo)
 * (Pillow's default quality is 75, OpenCV's 95).
 *   frames_dev    (N, h, w, 3) uint8 RGB on the device, h and w in 1..65535; quality in 1..100
 *   offsets_host  receives N + 1 byte offsets of the packed files (file k = [offsets[k], offsets[k+1]))
 * Encodes into the context's staging (grown when a call needs more): a counting pass gives the exact size of every file, `stream`
 * is synchronised, the offsets are written, and the files are written back to back behind their offsets on `stream`.
 */
int trs_jpeg_encode(trs_ctx* ctx, const uint8_t* frames_dev, int n, int h, int w, int quality, unsigned long long* offsets_host,
                    void* stream);
/* Copies the packed files of the last trs_jpeg_encode on this context (bytes must equal its offsets_host[n]) to blob_host
 * (pageable or pinned); call it on the stream of that encode.  Synchronises `stream`.  TRS_E_STATE: no encode yet. */
int trs_jpeg_encode_copy(trs_ctx* ctx, uint8_t* blob_host, unsigned long long bytes, void* stream);

/*
 * Forward pass of the pilots' networks (SURVEY.md 8(f) rank 4), replacing for N frames
 *   self.model(img_arr) / self.model((img_arr, spd)) / self.model((img_arr, spd, features))
 *                                           TritonRacerSim/components/keras_pilot.py:59,71,81,104
 * on the models built by
 *   Keras_2D_CNN.get_model                  TritonRacerSim/components/keras_train.py:127-174
 *   Keras_2D_FULL_HOUSE.get_model           TritonRacerSim/components/keras_train.py:184-245
 * together with the `np.asarray(img, float32) / 255` in front of them (keras_pilot.py:49-50).  Dropout is the identity at inference.
 * Arithmetic: tcgen05 tensor cores, fp16 operands (10-bit mantissa, as TensorFlow's TF32 convolutions on a GPU), fp32 accumulation,
 * fp16 activations between layers, fp32 in the Dense heads; not bit-exact with any CPU evaluation (tolerance: tests/test_pilot_gpu.py).
 *
 * Weights are host fp32 arrays in Keras layout, named "<layer>/kernel" (Conv2D: (kh, kw, in, out); Dense: (in, out)) and
 * "<layer>/bias" with the reference's layer names (conv1..conv7, dense1..dense3, output_layer, feature1..feature3; full house:
 * output_speed, current_spd_1..current_spd_3, dense4..dense6, out_steering).
 */
#define TRS_PILOT_CNN_2D 0             /* ModelType.CNN_2D          (utils/types.py): image -> (steering, throttle)          */
#define TRS_PILOT_CNN_2D_SPD_FTR 1     /* ModelType.CNN_2D_SPD_FTR : image + speed/20 -> (steering, throttle)                 */
#define TRS_PILOT_CNN_2D_SPD_CTL 2     /* ModelType.CNN_2D_SPD_CTL : image -> (steering, speed/20); same network as CNN_2D    */
#define TRS_PILOT_CNN_2D_FULL_HOUSE 3  /* ModelType.CNN_2D_FULL_HOUSE: image + speed/20 + loc/segment -> (steering, speed/20) */
typedef struct trs_pilot trs_pilot;
typedef struct trs_tensor {
    const char* name;
    const float* data;      /* host, C-contiguous */
    int32_t ndim;
    int32_t shape[4];
} trs_tensor;
/* h, w: frame size (w even, at least 93 x 93 so that every VALID convolution has an output); max_batch: frames per internal chunk
 * (sizes the activation workspace: about 0.6 MB per 120x160 frame; max_batch * h * w * 3 must stay below 4 GiB).
 * A trs_pilot owns one workspace: calls on the same pilot must be ordered (same stream, or synchronised by the caller); use one
 * pilot per stream for concurrent work.  trs_pilot_forward splits N into chunks of max_batch frames on the caller's stream. */
int trs_pilot_create(trs_ctx* ctx, int model_type, int h, int w, const trs_tensor* weights, int n_weights, int max_batch,
                     trs_pilot** out);
int trs_pilot_destroy(trs_pilot* p);
/*   frames_dev      (N,h,w,3) u8 `cam/img` / `cam/processed_img`
 *   spd_feature_dev (N) f32 gym/speed / 20   (SPD_FTR, FULL_HOUSE; keras_pilot.py:68,100-101)
 *   loc_feature_dev (N) f32 loc/segment      (FULL_HOUSE; keras_pilot.py:102-103)
 *   out_dev         (N,2) f32: the model's output row per frame */
int trs_pilot_forward(trs_pilot* p, const uint8_t* frames_dev, int n, const float* spd_feature_dev, const float* loc_feature_dev,
                      float* out_dev, void* stream);
/* The glue behind the model for ModelType.CNN_2D / CNN_2D_SPD_FTR (keras_pilot.py:59-63, 71-76): __cap on both outputs
 * (keras_pilot.py:142-145), __smooth_steering on the first (147-153), breaking = 0.0.  model_out_dev (N,2) f32; outputs (N) f64.
 * (CNN_2D_SPD_CTL / CNN_2D_FULL_HOUSE continue with trs_speed_control.) */
int trs_pilot_cap(trs_ctx* ctx, const float* model_out_dev, int n, int smooth_steering, double smooth_threshold, double* steering_dev,
                  double* throttle_dev, double* breaking_dev, void* stream);
/* Debug tap for the parity tests: activations of the most recent chunk.  layer 1..7: conv outputs, fp16
 * NHWC; 8: the fp32 partial sums of the first Dense layers.  Copies `bytes` bytes to host_out after synchronising `stream`. */
int trs_pilot_debug_activation(trs_pilot* p, int layer, void* host_out, unsigned long long bytes, void* stream);
/* Shape of a layer's output for one frame: (rows, cols, channels). */
int trs_pilot_layer_shape(trs_pilot* p, int layer, int* ho, int* wo, int* c);

/*
 * Host-buffer form of trs_preprocess: copies frames host->device in chunks, runs the kernels and
 * copies the requested outputs back, overlapping the three on internal streams; synchronises before
 * returning.  Host buffers may be pageable (slower) or pinned (trs_host_alloc).
 *   keep_f32_dev: optional device buffer (N,H,W,3) f32 that receives the normalised tensor and
 *   stays on the GPU for the pilot's model — nullable.
 *   stream: the caller's stream (cudaStream_t, NULL = the legacy default stream).  Work already queued on it
 *   (e.g. a pilot still reading keep_f32_dev from the previous step) is waited for before the internal
 *   streams touch any device buffer; everything is complete when the call returns, so the caller's stream
 *   may read keep_f32_dev right after it.
 */
int trs_preprocess_host(trs_ctx* ctx, const uint8_t* in_host, int n, int h, int w,
                        uint8_t* out_u8_host, float* out_f32_host, float* keep_f32_dev,
                        unsigned long long* stats_host, void* stream);

/*
 * Measurement aid (bench.py): the FP64 pipe rate of the context's GPU, the denominator of the nearest-waypoint kernel's roofline
 * (the scanning kernels behind trs_locate are FP64-ALU bound, SURVEY.md 8(d)).  dfma_tflops: dense DFMA chains, 2 flops per lane-instruction; dadd_tinst_per_s:
 * 10^12 DADD lane-instructions per second.  Synchronises.
 */
int trs_probe_fp64(trs_ctx* ctx, double* dfma_tflops, double* dadd_tinst_per_s);

/* Pinned host allocations for the *_host entry points. */
int trs_host_alloc(void** out, unsigned long long bytes);
int trs_host_free(void* p);

/* Debug taps used by the parity tests: intermediate planes of the edge filter for ONE frame.
 *   mag_dev (H,W) u16 selected-channel L1 magnitude; map_dev (H,W) u8: 0 none, 1 candidate, 2 strong. */
int trs_debug_canny_stages(trs_ctx* ctx, const uint8_t* in_dev, int h, int w,
                           uint16_t* mag_dev, uint8_t* map_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TRS_B200_H */
