/*
 * sgcore.h -- C ABI of the B200 spectrogram engine (libsgcore.so).
 *
 * This is the drop-in boundary for the frame-producing hot path of amilajack/spectrogram.
 * The reference delegates that path to the browser's AnalyserNode; the entry points below
 * are what a Node-API (or any FFI) binding for the path binds.  Each one cites the reference
 * interface it replaces (paths under the reference's src/).
 *
 * Conventions
 *   - plain C: pointers, sizes, POD structs; no C++/torch types cross this boundary
 *   - every function returns an sg_status (0 = ok, negative = error) unless noted;
 *     sg_last_error() returns a thread-local description of the last failure
 *   - Web Audio attribute violations map to SG_ERR_INDEX_SIZE (the binding throws
 *     IndexSizeError), wrong pointers/sizes to SG_ERR_INVALID_ARG (TypeError)
 *   - caller owns every output buffer; the engine borrows it for the duration of the call
 *     (javascripts/3D/visualizer.js:301 allocates the Uint8Array the reference passes in)
 *   - there is no CPU fallback: without a CUDA device sg_engine_create fails with
 *     SG_ERR_NO_DEVICE and nothing else can be called
 */
#ifndef SGCORE_H_
#define SGCORE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SG_VERSION_MAJOR 0
#define SG_VERSION_MINOR 1

typedef enum sg_status {
  SG_OK = 0,
  SG_ERR_INVALID_ARG = -1, /* null pointer, bad size, bad enum            -> TypeError        */
  SG_ERR_INDEX_SIZE = -2,  /* Web Audio IndexSizeError (fftSize, dB range, tau)               */
  SG_ERR_CUDA = -3,        /* a CUDA call failed; text in sg_last_error()                     */
  SG_ERR_OOM = -4,         /* device or pinned-host allocation failed                         */
  SG_ERR_NO_DEVICE = -5,   /* no usable CUDA device (there is no CPU fallback)                */
  SG_ERR_STATE = -6        /* call not valid in the object's current state                    */
} sg_status;

typedef enum sg_window {
  SG_WINDOW_BLACKMAN = 0, /* alpha = 0.16: what AnalyserNode applies (parity mode)            */
  SG_WINDOW_HANN = 1,     /* what BASELINE.json's configs name                                */
  SG_WINDOW_RECT = 2,
  SG_WINDOW_CUSTOM = 3    /* sg_stft_config.custom_window, n_fft floats                       */
} sg_window;

typedef enum sg_output {
  SG_OUT_U8 = 0,     /* getByteFrequencyData bytes        (3D/visualizer.js:352,358)          */
  SG_OUT_F32_DB = 1, /* getFloatFrequencyData dB, -inf for 0                                  */
  SG_OUT_RGBA8 = 2,  /* bytes through the sonogram colour LUT (bin/shaders/sonogram-*.shader) */
  SG_OUT_F32_MAG = 3 /* smoothed linear magnitude X^[k] (the analyser's internal state)       */
} sg_output;

typedef enum sg_align {
  SG_ALIGN_VALID = 0,   /* frame t = samples [t*hop, t*hop+n_fft); 1+(L-n_fft)/hop frames     */
  SG_ALIGN_ANALYSER = 1 /* frame t = the n_fft samples ending at (t+1)*hop, history starts
                           zero filled (AnalyserNode polled every `hop` samples); L/hop frames */
} sg_align;

/* Configuration of the batched path.  Replaces the reference's analyser configuration
 * (UI/player.js:7-11: fftSize, smoothingTimeConstant; defaults -100/-30 dB) plus the frame
 * cadence of UI/spectrogram.js:153-161 (one frame per requestAnimationFrame -> fixed hop). */
typedef struct sg_stft_config {
  int32_t n_fft;     /* even, 4..32768, n_fft/2 = 2^a 3^b 5^c; AnalyserNode objects need 2^k  */
  int32_t hop;       /* >= 1 samples between frames                                           */
  int32_t window;    /* sg_window                                                             */
  int32_t output;    /* sg_output                                                             */
  int32_t align;     /* sg_align                                                              */
  float min_db;      /* minDecibels, default -100                                             */
  float max_db;      /* maxDecibels, default -30; must be > min_db                            */
  float smoothing;   /* smoothingTimeConstant tau in [0,1]; state starts at 0 for every clip  */
  const float* custom_window; /* host pointer, n_fft floats, only for SG_WINDOW_CUSTOM        */
  const uint32_t* colormap;   /* host pointer, 256 RGBA8 (R | G<<8 | B<<16 | A<<24), or NULL
                                 for the reference's HSV map                                  */
} sg_stft_config;

typedef struct sg_engine sg_engine;     /* one per CUDA device; owns stream, plans, scratch   */
typedef struct sg_analyser sg_analyser; /* AnalyserNode-shaped single-stream object           */
typedef struct sg_stream sg_stream;     /* many concurrent channels, chunked (BASELINE cfg 5) */
typedef struct sg_ring sg_ring;         /* the reference's 256-row byte texture + its sonogram view */

/* ------------------------------------------------------------------ library ---------------- */
const char* sg_last_error(void);  /* thread-local, never NULL                                 */
int sg_version(void);             /* major*100 + minor                                        */
int sg_device_count(void);        /* number of CUDA devices visible, 0 if none                */

/* fills `cfg` with the reference's operating point: n_fft 2048 (UI/player.js:10), hop 512,
 * Blackman, u8 output, -100/-30 dB, tau 0 (UI/player.js:11), valid alignment */
int sg_stft_config_default(sg_stft_config* cfg);

/* ------------------------------------------------------------------ engine ----------------- */
int sg_engine_create(int device, sg_engine** out);
int sg_engine_destroy(sg_engine* e);
int sg_engine_device(const sg_engine* e);
/* number of kernels this engine has launched since creation (bench.py's gpu_launches) */
int64_t sg_engine_launch_count(const sg_engine* e);
/* name of the kernel family the last sg_stft_* call on this engine used
 * ("warp32x32x2p", "warp32x32x2", "warp32x32", "eo4096", "p16", "p8", "p4", "w16", "wreg", "r400", "smem") */
const char* sg_engine_last_kernel(const sg_engine* e);

/* ------------------------------------------------------------------ batched path ----------- */
/* frequencyBinCount (3D/visualizer.js:299,301): n_fft/2 */
int sg_stft_num_bins(const sg_stft_config* cfg);
/* frames produced for one clip of clip_len samples (<0: invalid cfg) */
int64_t sg_stft_num_frames(const sg_stft_config* cfg, int64_t clip_len);
/* bytes of one output element: 1 (u8) or 4 (f32, rgba8) */
int sg_stft_elem_bytes(const sg_stft_config* cfg);

/* Whole path on HOST buffers: pcm [n_clips][clip_len] float32 -> out [n_clips][frames][bins]
 * of the output element type.  Host->device and device->host copies happen inside the call
 * (staged through the engine's pinned buffers).  Replaces the reference's loop of
 * analyser.getByteFrequencyData(freqByteData) + texSubImage2D row append
 * (3D/visualizer.js:352-358, 399-416) for an offline clip. */
int sg_stft_batch(sg_engine* e, const float* pcm, int64_t n_clips, int64_t clip_len,
                  const sg_stft_config* cfg, void* out);

/* Clips sharded over several engines, one per GPU (SURVEY 8(e)): engine s takes the contiguous block of clips
 * [n_clips*s/G, n_clips*(s+1)/G); one host thread per engine inside the library runs sg_stft_batch's copy/compute
 * pipeline on its block and writes its results into its own slice of `out` -- that host copy is the gather, the
 * shards exchange nothing (no collective).  The result is bit-identical to sg_stft_batch on one engine.
 * Replaces, for a batch of offline clips, G independent copies of the reference's frame loop
 * (UI/spectrogram.js:153-161 + 3D/visualizer.js:399-416).  An engine may appear only once in the list. */
int sg_stft_batch_multi(sg_engine* const* engines, int n_engines, const float* pcm, int64_t n_clips,
                        int64_t clip_len, const sg_stft_config* cfg, void* out);

/* Same, on DEVICE-resident buffers, asynchronous on `cuda_stream` (a cudaStream_t / CUstream
 * handle; NULL = the engine's own stream).  clip_stride = samples between clip starts
 * (>= clip_len).  pcm_dev and out_dev must be 16-byte aligned.  Does not synchronise.
 * Calls with smoothing > 0 (or a custom colormap) share the engine's scratch buffers: the engine orders such a call
 * after the previous one with an event, whatever streams the two were given, so they serialise on the device. */
int sg_stft_batch_device(sg_engine* e, const float* pcm_dev, int64_t n_clips, int64_t clip_len,
                         int64_t clip_stride, const sg_stft_config* cfg, void* out_dev,
                         void* cuda_stream);

/* Kernel selection, for the parity tests (every kernel that can serve a shape is checked against the
 * oracle) and for A/B timing:  0 = automatic;  1 = generic shared-memory kernel for every shape;
 * 2 = n_fft 2048 on the one-frame-per-warp kernel;  3 = n_fft 2048 on the register family (wreg);
 * 4 = n_fft 2048 on the TMA-staged frame-pair kernel;
 * 6 = the register-pipelined frame-pair kernel with 8 instead of 12 warps per SM;
 * 7 = smoothingTimeConstant > 0 on the fused one-pass kernel of the shape (n_fft 256 ... 8192, hop <= n_fft) for ANY
 *     clip count, with chained segments (automatic selection runs one chain per clip from ~45 % of the co-resident CTA
 *     count in clips, independent segments with a warm-up below that when a segment is at least as long as its warm-up,
 *     and the two-kernel path otherwise).
 * 3 also selects the register family for n_fft 256 / 512 / 1024 (which have dedicated kernels by default). */
int sg_engine_set_kernel_variant(sg_engine* e, int variant);

/* page-locked host memory for the caller's input/output arrays: sg_stft_batch and sg_stream_push
 * DMA straight from/to such buffers and stage pageable ones through internal pinned buffers */
int sg_host_alloc(size_t bytes, void** out);
int sg_host_free(void* p);

/* waits for everything queued on the engine's own stream */
int sg_engine_synchronize(sg_engine* e);

/* the colour LUT the engine applies for SG_OUT_RGBA8 when cfg.colormap is NULL:
 * out = clamp(0.08 + a*HSV(360-360a, 1, 1)), a = byte/255, alpha 255
 * (bin/shaders/sonogram-vertex.shader:19-58, sonogram-fragment.shader:24-26,
 * background 3D/visualizer.js:69) */
int sg_colormap_reference(uint32_t lut[256]);

/* ------------------------------------------------------------------ AnalyserNode ----------- */
/* context.createAnalyser() (UI/player.js:7).  Defaults: fftSize 2048, -100/-30 dB, tau 0.8. */
int sg_analyser_create(sg_engine* e, sg_analyser** out);
int sg_analyser_destroy(sg_analyser* a);
/* analyser.fftSize = ... (UI/player.js:10): power of two in [32, 32768] else INDEX_SIZE */
int sg_analyser_set_fft_size(sg_analyser* a, int fft_size);
int sg_analyser_get_fft_size(const sg_analyser* a);
/* analyser.frequencyBinCount (3D/visualizer.js:299,301) */
int sg_analyser_get_frequency_bin_count(const sg_analyser* a);
int sg_analyser_set_min_decibels(sg_analyser* a, double v); /* must stay < maxDecibels        */
int sg_analyser_set_max_decibels(sg_analyser* a, double v); /* must stay > minDecibels        */
double sg_analyser_get_min_decibels(const sg_analyser* a);
double sg_analyser_get_max_decibels(const sg_analyser* a);
/* analyser.smoothingTimeConstant = ... (UI/player.js:11, 3D/visualizer.js:351,357,362) */
int sg_analyser_set_smoothing_time_constant(sg_analyser* a, double tau);
double sg_analyser_get_smoothing_time_constant(const sg_analyser* a);
/* Stands in for the audio render thread feeding the node (mix.connect(analyser),
 * UI/player.js:25): appends n mono samples to the node's ring. */
int sg_analyser_push(sg_analyser* a, const float* samples, int64_t n);
/* analyser.getByteFrequencyData(freqByteData) (3D/visualizer.js:352,358): writes
 * min(len, frequencyBinCount) bytes.  Advances the smoothing state once per push epoch
 * (two calls without a push in between return the same data). */
int sg_analyser_get_byte_frequency_data(sg_analyser* a, uint8_t* dst, int64_t len);
int sg_analyser_get_float_frequency_data(sg_analyser* a, float* dst, int64_t len);
/* analyser.getByteTimeDomainData(freqByteData) (3D/visualizer.js:363): min(len, fftSize) */
int sg_analyser_get_byte_time_domain_data(sg_analyser* a, uint8_t* dst, int64_t len);
int sg_analyser_get_float_time_domain_data(sg_analyser* a, float* dst, int64_t len);

/* ------------------------------------------------------------------ streaming -------------- */
/* n_channels independent AnalyserNode-like streams advanced in lock step (BASELINE config 5:
 * 256 channels, n_fft 1024, hop 128).  cfg.align is ignored (always analyser alignment);
 * cfg.output selects the primary output; max_chunk = the largest chunk_len push will see,
 * a multiple of cfg.hop. */
int sg_stream_create(sg_engine* e, int n_channels, const sg_stft_config* cfg, int max_chunk,
                     sg_stream** out);
int sg_stream_destroy(sg_stream* s);
int sg_stream_reset(sg_stream* s); /* zero history and smoothing state, and clear an attached sonogram history */
/* chunk: host [n_channels][chunk_len] float32, chunk_len a multiple of hop.
 * out: host [n_channels][chunk_len/hop][bins] elements of cfg.output.  It may be NULL when a
 * sonogram history is attached (sg_stream_set_history): the rows then only land in the history.
 * out_rgba (may be NULL): additionally host [n_channels][chunk_len/hop][bins] RGBA8 through the
 * colour LUT, cfg.colormap or the reference's when it is NULL (only when cfg.output == SG_OUT_U8,
 * and only with out).  Synchronous: returns when
 * both are filled and the history holds the new rows. */
int sg_stream_push(sg_stream* s, const float* chunk, int chunk_len, void* out, uint32_t* out_rgba);
int64_t sg_stream_frames_emitted(const sg_stream* s); /* per channel */
/* geometry of a stream object (any pointer may be NULL): what a binding needs to check the caller's array lengths */
int sg_stream_info(const sg_stream* s, int* channels, int* hop, int* bins, int* output, int* max_chunk);

/* Sonogram history of a stream: per channel, what an sg_ring(bins, rows) holds when it is fed
 * every push's byte rows, kept on the device and filled there (device-to-device) by each push.
 * Texture [n_channels][rows][bins] u8; the channels share one yoffset.  Needs cfg.output ==
 * SG_OUT_U8 (else SG_ERR_INVALID_ARG).  rows in [2, 65536], or 0 to detach (else
 * SG_ERR_INVALID_ARG).  Attaching, even with the current row count, starts it empty: texture
 * zero, yoffset 0 (initByteBuffer, visualizer.js:317-329). */
int sg_stream_set_history(sg_stream* s, int rows);
/* rows = 0 when no history is attached; either pointer may be NULL */
int sg_stream_history_info(const sg_stream* s, int* rows, int* yoffset);
/* channels [first, first+count) of the texture, host [count][rows][bins], texture row order
 * (each channel equals sg_ring_read of its ring) */
int sg_stream_history_read(sg_stream* s, int first, int count, uint8_t* dst);
/* sg_ring_view of channels [first, first+count) in one launch: host [count][height][width] RGBA8,
 * each image bit-identical to sg_ring_view of that channel's ring.  Page-locked rgba_out is
 * written by DMA directly.  Errors: SG_ERR_INVALID_ARG for a NULL pointer, width or height < 1,
 * width * height > 2^28, count * width * height > 2^30, or a channel range outside
 * [0, n_channels) or empty; then SG_ERR_STATE when no history is attached.  The same channel
 * range and state rules apply to sg_stream_history_read. */
int sg_stream_view(sg_stream* s, int first, int count, int width, int height, uint32_t* rgba_out);

/* ------------------------------------------------------------------ biquad filter ---------- */
/* W3C BiquadFilterNode.  The reference's draw mode (Player.setBandpassFrequency, UI/player.js) puts one in front of
 * the analyser: type 'bandpass', Q 10, frequency = the band under the pointer, so the sonogram shows only that band.
 *
 * Parameters: type (enum below, the spec's order), frequency (Hz, default 350), q (default 1), gain (dB, default 0),
 * detune (cents, default 0), sample_rate (the context's rate: an integer in [3000, 768000]).  A non-finite parameter, a
 * bad type or a bad sample_rate is SG_ERR_INVALID_ARG.  f0 = frequency * 2^(detune/1200) clamped to [0, sample_rate/2]
 * (frequency 0 stays 0 whatever the detune); q and gain take any finite value; gain only matters to lowshelf,
 * highshelf and peaking.
 *
 * Coefficients, in double: w0 = 2 pi f0/Fs, c = cos w0, A = 10^(gain/40);
 *   aQ = sin w0/(2 q)              (bandpass, notch, allpass, peaking)
 *   aQdB = sin w0/(2 10^(q/20))    (lowpass, highpass)
 *   aS = sin w0/sqrt(2)            (the shelves, S = 1)
 *   type       b0                       b1                  b2                       a0                     a1                   a2
 *   lowpass    (1-c)/2                  1-c                 (1-c)/2                  1+aQdB                 -2c                  1-aQdB
 *   highpass   (1+c)/2                  -(1+c)              (1+c)/2                  1+aQdB                 -2c                  1-aQdB
 *   bandpass   aQ                       0                   -aQ                      1+aQ                   -2c                  1-aQ
 *   lowshelf   A[(A+1)-(A-1)c+2aS vA]   2A[(A-1)-(A+1)c]    A[(A+1)-(A-1)c-2aS vA]   (A+1)+(A-1)c+2aS vA    -2[(A-1)+(A+1)c]     (A+1)+(A-1)c-2aS vA
 *   highshelf  A[(A+1)+(A-1)c+2aS vA]   -2A[(A-1)+(A+1)c]   A[(A+1)+(A-1)c-2aS vA]   (A+1)-(A-1)c+2aS vA    2[(A-1)-(A+1)c]      (A+1)-(A-1)c-2aS vA
 *   peaking    1+aQ A                   -2c                 1-aQ A                   1+aQ/A                 -2c                  1-aQ/A
 *   notch      1                        -2c                 1                        1+aQ                   -2c                  1-aQ
 *   allpass    1-aQ                     -2c                 1+aQ                     1+aQ                   -2c                  1-aQ
 * (vA = sqrt(A)), every coefficient divided by a0.  Where the formulas degenerate the filter is the limit of H(z), a
 * constant k (b0 = k, b1 = b2 = a1 = a2 = 0):
 *   f0 = 0:       lowpass, bandpass -> 0;  highpass, lowshelf, peaking, notch, allpass -> 1;  highshelf -> A^2
 *   f0 = Fs/2:    lowpass, highshelf, peaking, notch, allpass -> 1;  highpass, bandpass -> 0;  lowshelf -> A^2
 *   q <= 0 with 0 < f0 < Fs/2:  bandpass -> 1;  notch -> 0;  allpass -> -1;  peaking -> A^2
 *
 * Filtering is direct form I, y[n] = b0 x[n] + b1 x[n-1] + b2 x[n-2] - a1 y[n-1] - a2 y[n-2], with float64 arithmetic
 * and float64 state, each output rounded to float32 once.  Per channel the state is {x1, x2, y1, y2} (four doubles;
 * y unrounded).  The kernel runs each channel along time in parallel, which reorders the double arithmetic: every
 * output is within 1 float32 ulp of the sequential float64 recurrence rounded to float32, or within 2^-30 max|x| of
 * the channel, whichever is larger, also when a channel is split over calls with the state carried.  The launches
 * depend only on (n_channels, len), so equal inputs give bit-identical outputs.  Non-finite samples propagate as
 * IEEE arithmetic gives. */
typedef enum sg_biquad_type {
  SG_BIQUAD_LOWPASS = 0, SG_BIQUAD_HIGHPASS = 1, SG_BIQUAD_BANDPASS = 2, SG_BIQUAD_LOWSHELF = 3,
  SG_BIQUAD_HIGHSHELF = 4, SG_BIQUAD_PEAKING = 5, SG_BIQUAD_NOTCH = 6, SG_BIQUAD_ALLPASS = 7
} sg_biquad_type;

typedef struct sg_biquad_params {
  int32_t type;        /* sg_biquad_type                                                          */
  double sample_rate;  /* Hz, an integer in [3000, 768000]                                        */
  double frequency;    /* Hz                                                                      */
  double q;
  double gain;         /* dB                                                                      */
  double detune;       /* cents                                                                   */
} sg_biquad_params;

/* normalised {b0, b1, b2, a1, a2}; host only, needs no engine */
int sg_biquad_coefficients(const sg_biquad_params* p, double coef[5]);
/* in, out: host [n_channels][len] float32 (in == out allowed).  state: host [n_channels][4] doubles {x1, x2, y1, y2},
 * read as the initial state and written with the final one; NULL = zero start, no write-back.  Synchronous. */
int sg_biquad_filter(sg_engine* e, const sg_biquad_params* p, const float* in, int64_t n_channels, int64_t len,
                     double* state, float* out);
/* Same on device buffers, asynchronous on cuda_stream (NULL = the engine's stream); does not synchronise.  Channel c
 * reads in_dev + c*in_stride and writes out_dev + c*out_stride (strides >= len).  In place is allowed: in_dev == out_dev
 * with equal strides; otherwise the two must not overlap.  state_dev: device [n_channels][4] doubles, or NULL.
 * Channels longer than 4096 samples use three launches and the engine's scratch (ordered like sg_stft_batch_device's). */
int sg_biquad_filter_device(sg_engine* e, const sg_biquad_params* p, const float* in_dev, int64_t n_channels,
                            int64_t len, int64_t in_stride, float* out_dev, int64_t out_stride, double* state_dev,
                            void* cuda_stream);
/* The bank's filter (mix -> BiquadFilterNode -> analyser): with one attached, sg_stream_push filters each channel's new
 * chunk on the device, in place, before framing it.  NULL detaches the filter and drops its state.  The first attach
 * starts from zero state; changing the parameters while attached keeps the state (an AudioParam change between render
 * quanta, what dragging in draw mode does).  sg_stream_reset zeroes the state and keeps the parameters.  Works with any
 * cfg.output, with or without a sonogram history.  Errors as sg_biquad_coefficients. */
int sg_stream_set_filter(sg_stream* s, const sg_biquad_params* p);

/* ------------------------------------------------------------------ PCM ingestion ---------- */
/* The step in front of the path: the reference hands an encoded file to the browser,
 * context.decodeAudioData(request.response, buffer => ...) (util/util.js:9-17), plays the resulting
 * AudioBuffer through a buffer source (UI/player.js:110-115, 154-170) and the AnalyserNode down-mixes
 * whatever channels arrive to mono ([SPEC] AnalyserNode: "as if channelCount 1, channelCountMode max,
 * channelInterpretation speakers").  Built here for uncompressed PCM (RIFF/WAVE or raw interleaved
 * samples): sample-format conversion and the speakers down-mix run on the GPU, so 16-bit audio crosses
 * PCIe at 2 bytes per sample.  Compressed formats are NOT decoded.  decodeAudioData also resamples to the
 * context's rate; the *_resampled calls below do that on the GPU, fused with the conversion, with one fixed
 * filter: rational polyphase resampling equal to scipy.signal.resample_poly(x, up, down) with its default
 * Kaiser(beta 5) window (up/down = out_rate/in_rate reduced, half = 10*max(up, down), taps h[m] =
 * c sinc(c(m - half)) kaiser(m), c = 1/max(up, down), sum 1, times up; samples outside the clip are 0),
 * accumulated in float32.  Rates are integers in [3000, 768000] Hz and the reduced max(up, down) must be
 * <= 16384, else SG_ERR_INDEX_SIZE.  Equal rates take the plain ingest, bit for bit.  The other calls
 * carry sample_rate through unchanged. */
typedef enum sg_pcm_format {
  SG_PCM_U8 = 0,  /* unsigned 8 bit:            (v - 128) / 128                                 */
  SG_PCM_S16 = 1, /* little-endian signed 16:   v / 32768                                       */
  SG_PCM_S24 = 2, /* packed 3-byte signed:      v / 8388608                                     */
  SG_PCM_S32 = 3, /* signed 32:                 (float)v / 2147483648                           */
  SG_PCM_F32 = 4  /* IEEE float32, taken as is                                                  */
} sg_pcm_format;

typedef enum sg_pcm_layout {
  SG_PCM_MONO_MIX = 0, /* one plane: [SPEC] speakers down-mix to mono -- 1ch: x; 2ch: 0.5(L+R);
                          4ch: 0.25(L+R+SL+SR); 6ch: sqrt(1/2)(L+R) + C + 0.5(SL+SR); any other
                          count: discrete, i.e. channel 0                                        */
  SG_PCM_PLANAR = 1    /* `channels` planes (AudioBuffer.getChannelData(c)), analysed independently */
} sg_pcm_layout;

typedef struct sg_pcm_info {
  int32_t format;      /* sg_pcm_format                                                          */
  int32_t channels;    /* 1..32 interleaved channels                                             */
  int32_t sample_rate; /* Hz: the source rate of the *_resampled calls, informational elsewhere    */
  int64_t frames;      /* sample frames per clip (AudioBuffer.length)                            */
  int64_t data_offset; /* sg_wav_parse: byte offset of the first sample in the file; the ingest
                          calls take a pointer to the first sample and ignore this field         */
} sg_pcm_info;

/* bytes of one sample of `format` (1, 2, 3, 4, 4), 0 for a bad enum */
int sg_pcm_sample_bytes(int format);
/* planes the layout produces for `info`: 1 (mono mix) or info->channels (planar) */
int sg_pcm_num_planes(const sg_pcm_info* info, int layout);
/* Host-side RIFF/WAVE header walk (fmt + data chunks; PCM, IEEE float and WAVE_FORMAT_EXTENSIBLE).
 * Fills `out` (frames clipped to what the file actually holds).  No GPU involved. */
int sg_wav_parse(const void* file_bytes, size_t len, sg_pcm_info* out);
/* decodeAudioData for uncompressed PCM: n_clips clips of info->frames interleaved sample frames each,
 * back to back in host memory at `pcm`  ->  out host float32 [n_clips][planes][frames]. */
int sg_pcm_ingest(sg_engine* e, const void* pcm, int64_t n_clips, const sg_pcm_info* info, int layout,
                  float* out);
/* same on device buffers, asynchronous on cuda_stream (NULL = the engine's stream); plane p of clip c
 * is written at out_dev + (c*planes + p) * out_stride, out_stride >= info->frames floats */
int sg_pcm_ingest_device(sg_engine* e, const void* pcm_dev, int64_t n_clips, const sg_pcm_info* info,
                         int layout, float* out_dev, int64_t out_stride, void* cuda_stream);
/* Whole path from interleaved PCM on the host: ingest, then sg_stft_batch's pipeline with every plane a
 * clip.  out: host [n_clips][planes][frames_out][bins] of cfg->output.  The raw bytes (not float32) are
 * what crosses PCIe; copies, ingest and frame kernels overlap chunk by chunk. */
int sg_stft_pcm(sg_engine* e, const void* pcm, int64_t n_clips, const sg_pcm_info* info, int layout,
                const sg_stft_config* cfg, void* out);
/* frames after resampling `frames` from in_rate to out_rate: ceil(frames*up/down); <0 for invalid rates */
int64_t sg_resample_num_frames(int64_t frames, int32_t in_rate, int32_t out_rate);
/* sg_pcm_ingest, resampled from info->sample_rate to out_rate: out host [n_clips][planes][out_frames] */
int sg_pcm_ingest_resampled(sg_engine* e, const void* pcm, int64_t n_clips, const sg_pcm_info* info, int layout,
                            int32_t out_rate, float* out);
/* same on device buffers, asynchronous; plane p of clip c at out_dev + (c*planes+p)*out_stride, out_stride >= out_frames */
int sg_pcm_ingest_resampled_device(sg_engine* e, const void* pcm_dev, int64_t n_clips, const sg_pcm_info* info,
                                   int layout, int32_t out_rate, float* out_dev, int64_t out_stride, void* cuda_stream);
/* sg_stft_pcm with the planes resampled to out_rate before framing: out [n_clips][planes][frames(out_frames)][bins].
 * Bit-identical to sg_pcm_ingest_resampled followed by sg_stft_batch on the planes. */
int sg_stft_pcm_resampled(sg_engine* e, const void* pcm, int64_t n_clips, const sg_pcm_info* info, int layout,
                          int32_t out_rate, const sg_stft_config* cfg, void* out);

/* ------------------------------------------------------------------ sonogram ring + view --- */
/* The reference's spectrogram history: a bins x rows ALPHA/UNSIGNED_BYTE texture, one byte row per
 * frame written at yoffset, then yoffset = (yoffset + 1) % rows (3D/visualizer.js:60, 301-329,
 * 399-416; rows = 256 there).  Device resident: a streaming consumer appends rows and fetches the
 * rendered picture (or the raw texture) instead of re-uploading history. */
int sg_ring_create(sg_engine* e, int bins, int rows, sg_ring** out);
int sg_ring_destroy(sg_ring* r);
int sg_ring_reset(sg_ring* r); /* texture cleared to 0, yoffset 0 (initByteBuffer, visualizer.js:317-329) */
/* texSubImage2D of n_rows consecutive frames (host [n_rows][bins] u8), wrapping at `rows` */
int sg_ring_append(sg_ring* r, const uint8_t* frames, int n_rows);
int sg_ring_yoffset(const sg_ring* r);
int sg_ring_info(const sg_ring* r, int* bins, int* rows);   /* either pointer may be NULL */
/* the whole texture, host [rows][bins], in texture row order */
int sg_ring_read(sg_ring* r, uint8_t* dst);
/* Headless restatement of the sonogram view as an RGBA8 image, host [height][width]:
 * texCoord u = (px+.5)/width, v = (py+.5)/height; s = 256^(u-1) (log-frequency axis,
 * bin/shaders/sonogram-fragment.shader:16, sonogram-vertex.shader:51); t = v + yoffset/(rows-1)
 * (fragment:17, visualizer.js:460); a = LINEAR sample, CLAMP_TO_EDGE in s, REPEAT in t
 * (visualizer.js:312-315); colour HSV(360-360a,1,1) (sonogram-vertex.shader:19-58, per pixel);
 * fade sqrt(cos((1-v)pi/2)) (fragment:24); out = clamp(0.08 + a*fade*colour), alpha 255. */
int sg_ring_view(sg_ring* r, int width, int height, uint32_t* rgba_out);

#ifdef __cplusplus
}
#endif
#endif /* SGCORE_H_ */
