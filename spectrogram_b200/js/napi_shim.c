/*
 * napi_shim.c -- thin Node-API addon (spectrogram.node) over the C ABI in include/sgcore.h.
 *
 * This is the "thin C-ABI Node-API addon" BASELINE.json's north_star names: JavaScript host code
 * (index.js, an AnalyserNode-shaped facade) -> this shim -> libsgcore.so -> sm_100a kernels.
 * It contains no arithmetic: it unpacks JS arguments (numbers, option objects, typed arrays),
 * calls one sg_* function and maps sg_status to the exception a Web Audio host would see
 * (IndexSizeError -> RangeError with code 'IndexSizeError', bad arguments -> TypeError).
 * Typed arrays are borrowed for the duration of the call only (the reference allocates the
 * destination itself, src/javascripts/3D/visualizer.js:301, and passes it to
 * analyser.getByteFrequencyData, :352/:358).
 *
 * Node cannot run in this image; the shim is compiled against hand-declared prototypes
 * (node_api_min.h) and exercised by tests/napi_host/fake_napi_host.c, a C host that supplies the
 * napi_* symbols.  Under real Node the same object file loads unchanged.
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/sgcore.h"
#include "node_api_min.h"

#define MAX_ARGS 8

/* ---------------------------------------------------------------- helpers */
static napi_value undefined_of(napi_env env) {
  napi_value u;
  napi_get_undefined(env, &u);
  return u;
}

/* maps a failed sg_status to a pending JS exception; returns undefined */
static napi_value throw_status(napi_env env, int rc) {
  const char* msg = sg_last_error();
  if (rc == SG_ERR_INDEX_SIZE) napi_throw_range_error(env, "IndexSizeError", msg);
  else if (rc == SG_ERR_INVALID_ARG) napi_throw_type_error(env, "ERR_INVALID_ARG_TYPE", msg);
  else if (rc == SG_ERR_NO_DEVICE) napi_throw_error(env, "ERR_NO_CUDA_DEVICE", msg);
  else if (rc == SG_ERR_OOM) napi_throw_error(env, "ERR_OUT_OF_MEMORY", msg);
  else if (rc == SG_ERR_STATE) napi_throw_error(env, "InvalidStateError", msg);
  else napi_throw_error(env, "ERR_CUDA", msg);
  return undefined_of(env);
}

static napi_value type_error(napi_env env, const char* msg) {
  napi_throw_type_error(env, "ERR_INVALID_ARG_TYPE", msg);
  return undefined_of(env);
}

static size_t get_args(napi_env env, napi_callback_info info, napi_value* argv) {
  size_t argc = MAX_ARGS;
  napi_get_cb_info(env, info, &argc, argv, NULL, NULL);
  return argc;
}

static int get_external(napi_env env, napi_value v, void** out) {
  napi_valuetype t;
  if (napi_typeof(env, v, &t) != napi_ok || t != napi_external) return 0;
  return napi_get_value_external(env, v, out) == napi_ok && *out != NULL;
}

static int get_typed(napi_env env, napi_value v, napi_typedarray_type want, void** data, size_t* len) {
  bool is = false;
  napi_typedarray_type t;
  if (napi_is_typedarray(env, v, &is) != napi_ok || !is) return 0;
  if (napi_get_typedarray_info(env, v, &t, len, data, NULL, NULL) != napi_ok) return 0;
  if (want == napi_uint8_array && t == napi_uint8_clamped_array) return 1;
  return t == want;
}

static int is_undefined(napi_env env, napi_value v) {
  napi_valuetype t;
  return napi_typeof(env, v, &t) != napi_ok || t == napi_undefined || t == napi_null;
}

static int prop_double(napi_env env, napi_value obj, const char* name, double* out) {
  bool has = false;
  napi_value v;
  if (napi_has_named_property(env, obj, name, &has) != napi_ok || !has) return 0;
  if (napi_get_named_property(env, obj, name, &v) != napi_ok || is_undefined(env, v)) return 0;
  return napi_get_value_double(env, v, out) == napi_ok;
}

static int prop_string(napi_env env, napi_value obj, const char* name, char* buf, size_t n) {
  bool has = false;
  napi_value v;
  napi_valuetype t;
  size_t got = 0;
  if (napi_has_named_property(env, obj, name, &has) != napi_ok || !has) return 0;
  if (napi_get_named_property(env, obj, name, &v) != napi_ok) return 0;
  if (napi_typeof(env, v, &t) != napi_ok || t != napi_string) return 0;
  return napi_get_value_string_utf8(env, v, buf, n, &got) == napi_ok;
}

/* {fftSize, hop, window, output, align, minDecibels, maxDecibels, smoothingTimeConstant, colormap}
 * -> sg_stft_config.  Returns 0 and leaves a TypeError pending on a malformed object. */
static int parse_config(napi_env env, napi_value obj, sg_stft_config* cfg) {
  napi_valuetype t;
  double d;
  char s[32];
  sg_stft_config_default(cfg);
  if (is_undefined(env, obj)) return 1;
  if (napi_typeof(env, obj, &t) != napi_ok || t != napi_object) {
    type_error(env, "options must be an object");
    return 0;
  }
  if (prop_double(env, obj, "fftSize", &d)) cfg->n_fft = (d == (int32_t)d) ? (int32_t)d : -1;
  if (prop_double(env, obj, "hop", &d)) cfg->hop = (d == (int32_t)d) ? (int32_t)d : -1;
  if (prop_double(env, obj, "minDecibels", &d)) cfg->min_db = (float)d;
  if (prop_double(env, obj, "maxDecibels", &d)) cfg->max_db = (float)d;
  if (prop_double(env, obj, "smoothingTimeConstant", &d)) cfg->smoothing = (float)d;
  if (prop_string(env, obj, "window", s, sizeof s)) {
    if (!strcmp(s, "blackman")) cfg->window = SG_WINDOW_BLACKMAN;
    else if (!strcmp(s, "hann")) cfg->window = SG_WINDOW_HANN;
    else if (!strcmp(s, "rect")) cfg->window = SG_WINDOW_RECT;
    else { type_error(env, "unknown window"); return 0; }
  } else {
    bool has = false;
    napi_value v;
    void* data;
    size_t len;
    if (napi_has_named_property(env, obj, "window", &has) == napi_ok && has &&
        napi_get_named_property(env, obj, "window", &v) == napi_ok && !is_undefined(env, v)) {
      if (!get_typed(env, v, napi_float32_array, &data, &len) || (int64_t)len != cfg->n_fft) {
        type_error(env, "window must be a name or a Float32Array of fftSize entries");
        return 0;
      }
      cfg->window = SG_WINDOW_CUSTOM;
      cfg->custom_window = (const float*)data;
    }
  }
  if (prop_string(env, obj, "output", s, sizeof s)) {
    if (!strcmp(s, "u8") || !strcmp(s, "byte")) cfg->output = SG_OUT_U8;
    else if (!strcmp(s, "db") || !strcmp(s, "float")) cfg->output = SG_OUT_F32_DB;
    else if (!strcmp(s, "rgba") || !strcmp(s, "rgba8")) cfg->output = SG_OUT_RGBA8;
    else if (!strcmp(s, "mag")) cfg->output = SG_OUT_F32_MAG;
    else { type_error(env, "unknown output"); return 0; }
  }
  if (prop_string(env, obj, "align", s, sizeof s)) {
    if (!strcmp(s, "valid")) cfg->align = SG_ALIGN_VALID;
    else if (!strcmp(s, "analyser")) cfg->align = SG_ALIGN_ANALYSER;
    else { type_error(env, "unknown align"); return 0; }
  }
  {
    bool has = false;
    napi_value v;
    void* data;
    size_t len;
    if (napi_has_named_property(env, obj, "colormap", &has) == napi_ok && has &&
        napi_get_named_property(env, obj, "colormap", &v) == napi_ok && !is_undefined(env, v)) {
      if (!get_typed(env, v, napi_uint32_array, &data, &len) || len != 256) {
        type_error(env, "colormap must be a Uint32Array of 256 entries");
        return 0;
      }
      cfg->colormap = (const uint32_t*)data;
    }
  }
  return 1;
}

static napi_value make_int(napi_env env, int64_t v) {
  napi_value r;
  napi_create_int64(env, v, &r);
  return r;
}

/* ---------------------------------------------------------------- library / engine */
static napi_value js_device_count(napi_env env, napi_callback_info info) {
  (void)info;
  return make_int(env, sg_device_count());
}

static napi_value js_engine_create(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], r;
  size_t argc = get_args(env, info, argv);
  int32_t device = 0;
  sg_engine* e = NULL;
  int rc;
  if (argc >= 1 && !is_undefined(env, argv[0]) && napi_get_value_int32(env, argv[0], &device) != napi_ok)
    return type_error(env, "device must be an integer");
  rc = sg_engine_create(device, &e);
  if (rc != SG_OK) return throw_status(env, rc);
  napi_create_external(env, e, NULL, NULL, &r);
  return r;
}

static napi_value js_engine_destroy(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void* e;
  if (get_args(env, info, argv) < 1 || !get_external(env, argv[0], &e)) return type_error(env, "engine expected");
  sg_engine_destroy((sg_engine*)e);
  return undefined_of(env);
}

static napi_value js_engine_last_kernel(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], r;
  void* e;
  if (get_args(env, info, argv) < 1 || !get_external(env, argv[0], &e)) return type_error(env, "engine expected");
  napi_create_string_utf8(env, sg_engine_last_kernel((sg_engine*)e), NAPI_AUTO_LENGTH, &r);
  return r;
}

/* numFrames(options, clipLen) -> frames per clip; throws IndexSizeError on invalid attributes */
static napi_value js_num_frames(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  sg_stft_config cfg;
  int64_t clip_len = 0, n;
  if (get_args(env, info, argv) < 2) return type_error(env, "numFrames(options, clipLen)");
  if (!parse_config(env, argv[0], &cfg)) return undefined_of(env);
  if (napi_get_value_int64(env, argv[1], &clip_len) != napi_ok) return type_error(env, "clipLen must be a number");
  n = sg_stft_num_frames(&cfg, clip_len);
  if (n < 0) return throw_status(env, SG_ERR_INDEX_SIZE);
  return make_int(env, n);
}

/* stftBatch(engine, pcm: Float32Array, nClips, clipLen, options, out: Uint8Array|Float32Array|Uint32Array) */
static napi_value js_stft_batch(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *e, *pcm, *out;
  size_t pcm_len, out_len;
  int64_t n_clips, clip_len, frames;
  sg_stft_config cfg;
  napi_typedarray_type want;
  int rc;
  if (get_args(env, info, argv) < 6) return type_error(env, "stftBatch(engine, pcm, nClips, clipLen, options, out)");
  if (!get_external(env, argv[0], &e)) return type_error(env, "engine expected");
  if (!get_typed(env, argv[1], napi_float32_array, &pcm, &pcm_len)) return type_error(env, "pcm must be a Float32Array");
  if (napi_get_value_int64(env, argv[2], &n_clips) != napi_ok || napi_get_value_int64(env, argv[3], &clip_len) != napi_ok)
    return type_error(env, "nClips and clipLen must be numbers");
  if (!parse_config(env, argv[4], &cfg)) return undefined_of(env);
  if (n_clips < 0 || clip_len < 0 || (uint64_t)n_clips * (uint64_t)clip_len > pcm_len)
    return type_error(env, "pcm is shorter than nClips * clipLen");
  frames = sg_stft_num_frames(&cfg, clip_len);
  if (frames < 0) return throw_status(env, SG_ERR_INDEX_SIZE);
  want = cfg.output == SG_OUT_U8 ? napi_uint8_array : (cfg.output == SG_OUT_RGBA8 ? napi_uint32_array : napi_float32_array);
  if (!get_typed(env, argv[5], want, &out, &out_len)) return type_error(env, "out has the wrong typed-array type for this output");
  if ((uint64_t)out_len < (uint64_t)n_clips * (uint64_t)frames * (uint64_t)(cfg.n_fft / 2))
    return type_error(env, "out is shorter than nClips * frames * bins");
  rc = sg_stft_batch((sg_engine*)e, (const float*)pcm, n_clips, clip_len, &cfg, out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* stftBatchMulti(engines: [engine, ...], pcm, nClips, clipLen, options, out): clips sharded over the engines in
 * contiguous blocks inside the library (one host thread per engine), results gathered into `out` */
static napi_value js_stft_batch_multi(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], item;
  sg_engine* engines[64];
  void *e, *pcm, *out;
  size_t pcm_len, out_len;
  uint32_t n_eng = 0, i;
  int64_t n_clips, clip_len, frames;
  sg_stft_config cfg;
  napi_typedarray_type want;
  bool is_arr = false;
  int rc;
  if (get_args(env, info, argv) < 6) return type_error(env, "stftBatchMulti(engines, pcm, nClips, clipLen, options, out)");
  if (napi_is_array(env, argv[0], &is_arr) != napi_ok || !is_arr || napi_get_array_length(env, argv[0], &n_eng) != napi_ok ||
      n_eng < 1 || n_eng > 64)
    return type_error(env, "engines must be an array of 1..64 engines");
  for (i = 0; i < n_eng; ++i) {
    if (napi_get_element(env, argv[0], i, &item) != napi_ok || !get_external(env, item, &e)) return type_error(env, "engine expected");
    engines[i] = (sg_engine*)e;
  }
  if (!get_typed(env, argv[1], napi_float32_array, &pcm, &pcm_len)) return type_error(env, "pcm must be a Float32Array");
  if (napi_get_value_int64(env, argv[2], &n_clips) != napi_ok || napi_get_value_int64(env, argv[3], &clip_len) != napi_ok)
    return type_error(env, "nClips and clipLen must be numbers");
  if (!parse_config(env, argv[4], &cfg)) return undefined_of(env);
  if (n_clips < 0 || clip_len < 0 || (uint64_t)n_clips * (uint64_t)clip_len > pcm_len)
    return type_error(env, "pcm is shorter than nClips * clipLen");
  frames = sg_stft_num_frames(&cfg, clip_len);
  if (frames < 0) return throw_status(env, SG_ERR_INDEX_SIZE);
  want = cfg.output == SG_OUT_U8 ? napi_uint8_array : (cfg.output == SG_OUT_RGBA8 ? napi_uint32_array : napi_float32_array);
  if (!get_typed(env, argv[5], want, &out, &out_len)) return type_error(env, "out has the wrong typed-array type for this output");
  if ((uint64_t)out_len < (uint64_t)n_clips * (uint64_t)frames * (uint64_t)(cfg.n_fft / 2))
    return type_error(env, "out is shorter than nClips * frames * bins");
  rc = sg_stft_batch_multi(engines, (int)n_eng, (const float*)pcm, n_clips, clip_len, &cfg, out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

static napi_value js_colormap_reference(napi_env env, napi_callback_info info) {
  napi_value ab, ta;
  void* data = NULL;
  (void)info;
  if (napi_create_arraybuffer(env, 256 * sizeof(uint32_t), &data, &ab) != napi_ok || !data)
    return type_error(env, "could not allocate the colour table");
  sg_colormap_reference((uint32_t*)data);
  napi_create_typedarray(env, napi_uint32_array, 256, ab, 0, &ta);
  return ta;
}

/* ---------------------------------------------------------------- AnalyserNode */
static napi_value js_analyser_create(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], r;
  void* e;
  sg_analyser* a = NULL;
  int rc;
  if (get_args(env, info, argv) < 1 || !get_external(env, argv[0], &e)) return type_error(env, "engine expected");
  rc = sg_analyser_create((sg_engine*)e, &a);
  if (rc != SG_OK) return throw_status(env, rc);
  napi_create_external(env, a, NULL, NULL, &r);
  return r;
}

static napi_value js_analyser_destroy(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void* a;
  if (get_args(env, info, argv) < 1 || !get_external(env, argv[0], &a)) return type_error(env, "analyser expected");
  sg_analyser_destroy((sg_analyser*)a);
  return undefined_of(env);
}

/* analyserSet(a, name, value): fftSize | minDecibels | maxDecibels | smoothingTimeConstant */
static napi_value js_analyser_set(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void* a;
  char name[32];
  size_t got;
  double v;
  int rc;
  if (get_args(env, info, argv) < 3 || !get_external(env, argv[0], &a)) return type_error(env, "analyserSet(analyser, name, value)");
  if (napi_get_value_string_utf8(env, argv[1], name, sizeof name, &got) != napi_ok) return type_error(env, "name must be a string");
  if (napi_get_value_double(env, argv[2], &v) != napi_ok) return type_error(env, "value must be a number");
  if (!strcmp(name, "fftSize")) rc = (v == (int)v) ? sg_analyser_set_fft_size((sg_analyser*)a, (int)v) : sg_analyser_set_fft_size((sg_analyser*)a, -1);
  else if (!strcmp(name, "minDecibels")) rc = sg_analyser_set_min_decibels((sg_analyser*)a, v);
  else if (!strcmp(name, "maxDecibels")) rc = sg_analyser_set_max_decibels((sg_analyser*)a, v);
  else if (!strcmp(name, "smoothingTimeConstant")) rc = sg_analyser_set_smoothing_time_constant((sg_analyser*)a, v);
  else return type_error(env, "unknown attribute");
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

static napi_value js_analyser_get(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], r;
  void* a;
  char name[32];
  size_t got;
  double v;
  if (get_args(env, info, argv) < 2 || !get_external(env, argv[0], &a)) return type_error(env, "analyserGet(analyser, name)");
  if (napi_get_value_string_utf8(env, argv[1], name, sizeof name, &got) != napi_ok) return type_error(env, "name must be a string");
  if (!strcmp(name, "fftSize")) v = sg_analyser_get_fft_size((sg_analyser*)a);
  else if (!strcmp(name, "frequencyBinCount")) v = sg_analyser_get_frequency_bin_count((sg_analyser*)a);
  else if (!strcmp(name, "minDecibels")) v = sg_analyser_get_min_decibels((sg_analyser*)a);
  else if (!strcmp(name, "maxDecibels")) v = sg_analyser_get_max_decibels((sg_analyser*)a);
  else if (!strcmp(name, "smoothingTimeConstant")) v = sg_analyser_get_smoothing_time_constant((sg_analyser*)a);
  else return type_error(env, "unknown attribute");
  napi_create_double(env, v, &r);
  return r;
}

static napi_value js_analyser_push(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *a, *data;
  size_t len;
  int rc;
  if (get_args(env, info, argv) < 2 || !get_external(env, argv[0], &a)) return type_error(env, "analyserPush(analyser, samples)");
  if (!get_typed(env, argv[1], napi_float32_array, &data, &len)) return type_error(env, "samples must be a Float32Array");
  rc = sg_analyser_push((sg_analyser*)a, (const float*)data, (int64_t)len);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

typedef int (*getter_u8)(sg_analyser*, uint8_t*, int64_t);
typedef int (*getter_f32)(sg_analyser*, float*, int64_t);

static napi_value analyser_read(napi_env env, napi_callback_info info, napi_typedarray_type want, getter_u8 g8, getter_f32 g32) {
  napi_value argv[MAX_ARGS];
  void *a, *data;
  size_t len;
  int rc;
  if (get_args(env, info, argv) < 2 || !get_external(env, argv[0], &a)) return type_error(env, "analyser expected");
  if (!get_typed(env, argv[1], want, &data, &len))
    return type_error(env, want == napi_uint8_array ? "a Uint8Array is required" : "a Float32Array is required");
  rc = g8 ? g8((sg_analyser*)a, (uint8_t*)data, (int64_t)len) : g32((sg_analyser*)a, (float*)data, (int64_t)len);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}
static napi_value js_get_byte_frequency_data(napi_env env, napi_callback_info info) {
  return analyser_read(env, info, napi_uint8_array, sg_analyser_get_byte_frequency_data, NULL);
}
static napi_value js_get_float_frequency_data(napi_env env, napi_callback_info info) {
  return analyser_read(env, info, napi_float32_array, NULL, sg_analyser_get_float_frequency_data);
}
static napi_value js_get_byte_time_domain_data(napi_env env, napi_callback_info info) {
  return analyser_read(env, info, napi_uint8_array, sg_analyser_get_byte_time_domain_data, NULL);
}
static napi_value js_get_float_time_domain_data(napi_env env, napi_callback_info info) {
  return analyser_read(env, info, napi_float32_array, NULL, sg_analyser_get_float_time_domain_data);
}

/* ---------------------------------------------------------------- streaming */
static napi_value js_stream_create(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], r;
  void* e;
  int32_t channels, max_chunk;
  sg_stft_config cfg;
  sg_stream* s = NULL;
  int rc;
  if (get_args(env, info, argv) < 4 || !get_external(env, argv[0], &e)) return type_error(env, "streamCreate(engine, channels, options, maxChunk)");
  if (napi_get_value_int32(env, argv[1], &channels) != napi_ok || napi_get_value_int32(env, argv[3], &max_chunk) != napi_ok)
    return type_error(env, "channels and maxChunk must be integers");
  if (!parse_config(env, argv[2], &cfg)) return undefined_of(env);
  rc = sg_stream_create((sg_engine*)e, channels, &cfg, max_chunk, &s);
  if (rc != SG_OK) return throw_status(env, rc);
  napi_create_external(env, s, NULL, NULL, &r);
  return r;
}

/* streamPush(stream, chunk: Float32Array, chunkLen, out | undefined, outRgba | undefined); out may be undefined only
 * when a sonogram history is attached (the rows then only land in the history) */
static napi_value js_stream_push(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *s, *chunk, *out = NULL, *rgba = NULL;
  size_t chunk_n, out_n = 0, rgba_n;
  int32_t chunk_len;
  bool is = false;
  int rc, have_out;
  size_t argc = get_args(env, info, argv);
  if (argc < 4 || !get_external(env, argv[0], &s)) return type_error(env, "streamPush(stream, chunk, chunkLen, out[, outRgba])");
  if (!get_typed(env, argv[1], napi_float32_array, &chunk, &chunk_n)) return type_error(env, "chunk must be a Float32Array");
  if (napi_get_value_int32(env, argv[2], &chunk_len) != napi_ok) return type_error(env, "chunkLen must be an integer");
  have_out = !is_undefined(env, argv[3]);
  if (have_out && (napi_is_typedarray(env, argv[3], &is) != napi_ok || !is ||
                   napi_get_typedarray_info(env, argv[3], NULL, &out_n, &out, NULL, NULL) != napi_ok))
    return type_error(env, "out must be a typed array");
  if (argc >= 5 && !is_undefined(env, argv[4]) && !get_typed(env, argv[4], napi_uint32_array, &rgba, &rgba_n))
    return type_error(env, "outRgba must be a Uint32Array");
  {
    /* the core reads channels * chunkLen samples and writes channels * (chunkLen / hop) * bins elements: check the
     * caller's arrays against the stream's own geometry before handing raw pointers over */
    int channels = 0, hop = 1, bins = 0, output = 0, max_chunk = 0;
    napi_typedarray_type got = napi_uint8_array;
    uint64_t need;
    if (sg_stream_info((sg_stream*)s, &channels, &hop, &bins, &output, &max_chunk) != SG_OK) return type_error(env, "stream expected");
    if (chunk_len < 0 || chunk_len > max_chunk || chunk_len % hop) return type_error(env, "chunkLen must be a multiple of hop, at most maxChunk");
    if ((uint64_t)chunk_n < (uint64_t)channels * (uint64_t)chunk_len) return type_error(env, "chunk is shorter than channels * chunkLen");
    need = (uint64_t)channels * (uint64_t)(chunk_len / hop) * (uint64_t)bins;
    if (have_out) {
      napi_get_typedarray_info(env, argv[3], &got, NULL, NULL, NULL, NULL);
      if (got != (output == SG_OUT_U8 ? napi_uint8_array : (output == SG_OUT_RGBA8 ? napi_uint32_array : napi_float32_array)))
        return type_error(env, "out has the wrong typed-array type for this stream's output");
      if ((uint64_t)out_n < need) return type_error(env, "out is shorter than channels * frames * bins");
      if (rgba && (uint64_t)rgba_n < need) return type_error(env, "outRgba is shorter than channels * frames * bins");
    } else {
      int rows = 0;
      if (sg_stream_history_info((sg_stream*)s, &rows, NULL) != SG_OK || !rows)
        return type_error(env, "out must be a typed array (it may be undefined only when a history is attached)");
      if (rgba) return type_error(env, "outRgba needs out");
    }
  }
  rc = sg_stream_push((sg_stream*)s, (const float*)chunk, chunk_len, out, (uint32_t*)rgba);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* streamSetHistory(stream, rows): attach an empty sonogram history of rows rows per channel, or detach it (rows 0) */
static napi_value js_stream_set_history(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void* s;
  int32_t rows;
  int rc;
  if (get_args(env, info, argv) < 2 || !get_external(env, argv[0], &s)) return type_error(env, "streamSetHistory(stream, rows)");
  if (napi_get_value_int32(env, argv[1], &rows) != napi_ok) return type_error(env, "rows must be an integer");
  rc = sg_stream_set_history((sg_stream*)s, rows);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* streamHistoryInfo(stream) -> {rows, yoffset}; rows is 0 when no history is attached */
static napi_value js_stream_history_info(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], o;
  void* s;
  int rows = 0, yoffset = 0;
  if (get_args(env, info, argv) < 1 || !get_external(env, argv[0], &s)) return type_error(env, "stream expected");
  if (sg_stream_history_info((sg_stream*)s, &rows, &yoffset) != SG_OK) return type_error(env, "stream expected");
  napi_create_object(env, &o);
  napi_set_named_property(env, o, "rows", make_int(env, rows));
  napi_set_named_property(env, o, "yoffset", make_int(env, yoffset));
  return o;
}

/* channels [first, first+count) of a stream's history checked against its geometry; 0 and a pending TypeError when the
 * range is outside the bank.  *rows and *bins get the texture's size (rows 0: no history; the core then reports it). */
static int history_range(napi_env env, void* s, int32_t first, int32_t count, int* rows, int* bins) {
  int channels = 0;
  if (sg_stream_info((sg_stream*)s, &channels, NULL, bins, NULL, NULL) != SG_OK ||
      sg_stream_history_info((sg_stream*)s, rows, NULL) != SG_OK) {
    type_error(env, "stream expected");
    return 0;
  }
  if (first < 0 || count < 1 || count > channels - first) {
    type_error(env, "channel range outside the bank");
    return 0;
  }
  return 1;
}

/* streamHistoryRead(stream, first, count, out: Uint8Array [count][rows][bins]) */
static napi_value js_stream_history_read(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *s, *out;
  size_t n;
  int32_t first, count;
  int rows = 0, bins = 0, rc;
  if (get_args(env, info, argv) < 4 || !get_external(env, argv[0], &s)) return type_error(env, "streamHistoryRead(stream, first, count, out)");
  if (napi_get_value_int32(env, argv[1], &first) != napi_ok || napi_get_value_int32(env, argv[2], &count) != napi_ok)
    return type_error(env, "first and count must be integers");
  if (!get_typed(env, argv[3], napi_uint8_array, &out, &n)) return type_error(env, "out must be a Uint8Array");
  if (!history_range(env, s, first, count, &rows, &bins)) return undefined_of(env);
  if ((uint64_t)n < (uint64_t)count * (uint64_t)rows * (uint64_t)bins) return type_error(env, "out is shorter than count * rows * bins");
  rc = sg_stream_history_read((sg_stream*)s, first, count, (uint8_t*)out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* streamView(stream, first, count, width, height, out: Uint32Array [count][height][width]): every channel's sonogram
 * picture in one launch */
static napi_value js_stream_view(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *s, *out;
  size_t n;
  int32_t first, count, w, h;
  int rows = 0, bins = 0, rc;
  if (get_args(env, info, argv) < 6 || !get_external(env, argv[0], &s)) return type_error(env, "streamView(stream, first, count, width, height, out)");
  if (napi_get_value_int32(env, argv[1], &first) != napi_ok || napi_get_value_int32(env, argv[2], &count) != napi_ok ||
      napi_get_value_int32(env, argv[3], &w) != napi_ok || napi_get_value_int32(env, argv[4], &h) != napi_ok)
    return type_error(env, "first, count, width and height must be integers");
  if (!get_typed(env, argv[5], napi_uint32_array, &out, &n)) return type_error(env, "out must be a Uint32Array");
  if (w < 1 || h < 1 || (uint64_t)w * (uint64_t)h > (1ull << 28)) return type_error(env, "image size out of range");
  if (!history_range(env, s, first, count, &rows, &bins)) return undefined_of(env);
  if ((uint64_t)n < (uint64_t)count * (uint64_t)w * (uint64_t)h) return type_error(env, "out is shorter than count * width * height");
  rc = sg_stream_view((sg_stream*)s, first, count, w, h, (uint32_t*)out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

static napi_value js_stream_destroy(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void* s;
  if (get_args(env, info, argv) < 1 || !get_external(env, argv[0], &s)) return type_error(env, "stream expected");
  sg_stream_destroy((sg_stream*)s);
  return undefined_of(env);
}

/* ---------------------------------------------------------------- biquad filter */
static const char* const kBiquadNames[8] = {"lowpass", "highpass", "bandpass", "lowshelf", "highshelf", "peaking", "notch", "allpass"};

/* {type, sampleRate, frequency, Q, gain, detune} -> sg_biquad_params; absent members take the BiquadFilterNode defaults
 * (lowpass, 48000, 350, 1, 0, 0).  Returns 0 and leaves a TypeError pending on a non-object or an unknown type (the JS
 * facade never sends one: it ignores such assignments, as WebIDL does for an enum attribute). */
static int parse_biquad(napi_env env, napi_value obj, sg_biquad_params* p) {
  napi_valuetype t;
  char s[32];
  int i;
  p->type = SG_BIQUAD_LOWPASS; p->sample_rate = 48000.0; p->frequency = 350.0; p->q = 1.0; p->gain = 0.0; p->detune = 0.0;
  if (napi_typeof(env, obj, &t) != napi_ok || t != napi_object) {
    type_error(env, "filter parameters must be an object");
    return 0;
  }
  prop_double(env, obj, "sampleRate", &p->sample_rate);
  prop_double(env, obj, "frequency", &p->frequency);
  prop_double(env, obj, "Q", &p->q);
  prop_double(env, obj, "gain", &p->gain);
  prop_double(env, obj, "detune", &p->detune);
  if (prop_string(env, obj, "type", s, sizeof s)) {
    for (i = 0; i < 8 && strcmp(s, kBiquadNames[i]); ++i) {}
    if (i == 8) {
      type_error(env, "unknown biquad type");
      return 0;
    }
    p->type = i;
  }
  return 1;
}

/* biquadCoefficients(params, out: Float64Array >= 5) -> normalised b0, b1, b2, a1, a2 */
static napi_value js_biquad_coefficients(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  sg_biquad_params p;
  void* out;
  size_t n;
  int rc;
  if (get_args(env, info, argv) < 2) return type_error(env, "biquadCoefficients(params, out)");
  if (!parse_biquad(env, argv[0], &p)) return undefined_of(env);
  if (!get_typed(env, argv[1], napi_float64_array, &out, &n) || n < 5) return type_error(env, "out must be a Float64Array of 5 entries");
  rc = sg_biquad_coefficients(&p, (double*)out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* biquadFilter(engine, params, samples: Float32Array [channels][len], channels, len, state: Float64Array [channels][4] |
 * undefined, out: Float32Array [channels][len]) */
static napi_value js_biquad_filter(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  sg_biquad_params p;
  void *e, *in, *out, *state = NULL;
  size_t in_n, out_n, state_n = 0;
  int64_t channels, len;
  uint64_t need;
  int rc;
  if (get_args(env, info, argv) < 7 || !get_external(env, argv[0], &e))
    return type_error(env, "biquadFilter(engine, params, samples, channels, len, state, out)");
  if (!parse_biquad(env, argv[1], &p)) return undefined_of(env);
  if (!get_typed(env, argv[2], napi_float32_array, &in, &in_n)) return type_error(env, "samples must be a Float32Array");
  if (napi_get_value_int64(env, argv[3], &channels) != napi_ok || napi_get_value_int64(env, argv[4], &len) != napi_ok ||
      channels < 0 || len < 0)
    return type_error(env, "channels and len must be non-negative integers");
  if (!is_undefined(env, argv[5]) && !get_typed(env, argv[5], napi_float64_array, &state, &state_n))
    return type_error(env, "state must be a Float64Array or undefined");
  if (!get_typed(env, argv[6], napi_float32_array, &out, &out_n)) return type_error(env, "out must be a Float32Array");
  /* the core reads and writes channels * len samples and channels * 4 state values: check before any pointer goes over */
  if (channels > 0 && (uint64_t)len > UINT64_MAX / (uint64_t)channels) return type_error(env, "channels * len overflows");
  need = (uint64_t)channels * (uint64_t)len;
  if ((uint64_t)in_n < need) return type_error(env, "samples is shorter than channels * len");
  if ((uint64_t)out_n < need) return type_error(env, "out is shorter than channels * len");
  if (state && (uint64_t)state_n < 4 * (uint64_t)channels) return type_error(env, "state is shorter than channels * 4");
  rc = sg_biquad_filter((sg_engine*)e, &p, (const float*)in, channels, len, (double*)state, (float*)out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* streamSetFilter(stream, params | null | undefined): attach or retune the bank's filter; null detaches it */
static napi_value js_stream_set_filter(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  sg_biquad_params p;
  void* s;
  int rc, channels = 0;
  if (get_args(env, info, argv) < 2 || !get_external(env, argv[0], &s)) return type_error(env, "streamSetFilter(stream, params)");
  if (sg_stream_info((sg_stream*)s, &channels, NULL, NULL, NULL, NULL) != SG_OK) return type_error(env, "stream expected");
  if (!is_undefined(env, argv[1]) && !parse_biquad(env, argv[1], &p)) return undefined_of(env);
  rc = sg_stream_set_filter((sg_stream*)s, is_undefined(env, argv[1]) ? NULL : &p);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* ---------------------------------------------------------------- sonogram ring + view */
/* ringCreate(engine, bins, rows): the reference's bins x 256 byte texture (3D/visualizer.js:301-329) */
static napi_value js_ring_create(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], r;
  void* e;
  int32_t bins, rows;
  sg_ring* ring = NULL;
  int rc;
  if (get_args(env, info, argv) < 3 || !get_external(env, argv[0], &e)) return type_error(env, "ringCreate(engine, bins, rows)");
  if (napi_get_value_int32(env, argv[1], &bins) != napi_ok || napi_get_value_int32(env, argv[2], &rows) != napi_ok)
    return type_error(env, "bins and rows must be integers");
  rc = sg_ring_create((sg_engine*)e, bins, rows, &ring);
  if (rc != SG_OK) return throw_status(env, rc);
  napi_create_external(env, ring, NULL, NULL, &r);
  return r;
}

/* ringAppend(ring, frames: Uint8Array, nRows): texSubImage2D at yoffset + advance (visualizer.js:399-416) */
static napi_value js_ring_append(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *ring, *frames;
  size_t n;
  int32_t n_rows;
  int rc;
  if (get_args(env, info, argv) < 3 || !get_external(env, argv[0], &ring)) return type_error(env, "ringAppend(ring, frames, nRows)");
  if (!get_typed(env, argv[1], napi_uint8_array, &frames, &n)) return type_error(env, "frames must be a Uint8Array");
  if (napi_get_value_int32(env, argv[2], &n_rows) != napi_ok) return type_error(env, "nRows must be an integer");
  {
    int bins = 0;
    if (sg_ring_info((sg_ring*)ring, &bins, NULL) != SG_OK) return type_error(env, "ring expected");
    if (n_rows < 0 || (uint64_t)n < (uint64_t)n_rows * (uint64_t)bins) return type_error(env, "frames is shorter than nRows * bins");
  }
  rc = sg_ring_append((sg_ring*)ring, (const uint8_t*)frames, n_rows);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

static napi_value js_ring_yoffset(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void* ring;
  if (get_args(env, info, argv) < 1 || !get_external(env, argv[0], &ring)) return type_error(env, "ring expected");
  return make_int(env, sg_ring_yoffset((sg_ring*)ring));
}

/* ringView(ring, width, height, out: Uint32Array): the sonogram picture (sonogram-fragment.shader:14-27) */
static napi_value js_ring_view(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *ring, *out;
  size_t n;
  int32_t w, h;
  int rc;
  if (get_args(env, info, argv) < 4 || !get_external(env, argv[0], &ring)) return type_error(env, "ringView(ring, width, height, out)");
  if (napi_get_value_int32(env, argv[1], &w) != napi_ok || napi_get_value_int32(env, argv[2], &h) != napi_ok)
    return type_error(env, "width and height must be integers");
  if (!get_typed(env, argv[3], napi_uint32_array, &out, &n)) return type_error(env, "out must be a Uint32Array");
  if (w < 1 || h < 1 || n < (size_t)w * (size_t)h) return type_error(env, "out is smaller than width * height");
  rc = sg_ring_view((sg_ring*)ring, w, h, (uint32_t*)out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

static napi_value js_ring_destroy(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void* ring;
  if (get_args(env, info, argv) < 1 || !get_external(env, argv[0], &ring)) return type_error(env, "ring expected");
  sg_ring_destroy((sg_ring*)ring);
  return undefined_of(env);
}

/* ---------------------------------------------------------------- PCM ingestion (decodeAudioData for PCM) */
static const char* const kPcmNames[5] = {"u8", "s16", "s24", "s32", "f32"};

/* wavParse(file: Uint8Array) -> {format, channels, sampleRate, length, dataOffset}: the header walk in front of
 * context.decodeAudioData (util/util.js:9); host only */
static napi_value js_wav_parse(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], o, v;
  void* bytes;
  size_t n;
  sg_pcm_info pi;
  int rc;
  if (get_args(env, info, argv) < 1 || !get_typed(env, argv[0], napi_uint8_array, &bytes, &n))
    return type_error(env, "wavParse(file: Uint8Array)");
  rc = sg_wav_parse(bytes, n, &pi);
  if (rc != SG_OK) return throw_status(env, rc);
  napi_create_object(env, &o);
  napi_create_string_utf8(env, kPcmNames[pi.format], NAPI_AUTO_LENGTH, &v); napi_set_named_property(env, o, "format", v);
  napi_create_int32(env, pi.channels, &v); napi_set_named_property(env, o, "channels", v);
  napi_create_int32(env, pi.sample_rate, &v); napi_set_named_property(env, o, "sampleRate", v);
  napi_create_double(env, (double)pi.frames, &v); napi_set_named_property(env, o, "length", v);
  napi_create_double(env, (double)pi.data_offset, &v); napi_set_named_property(env, o, "dataOffset", v);
  return o;
}

/* {format, channels, sampleRate} + the byte length of `samples` -> sg_pcm_info for n_clips clips */
static int parse_pcm(napi_env env, napi_value obj, size_t n_bytes, int32_t n_clips, sg_pcm_info* pi) {
  napi_valuetype t;
  double d;
  char s[8];
  int bpf;
  memset(pi, 0, sizeof *pi);
  pi->format = -1;
  if (napi_typeof(env, obj, &t) != napi_ok || t != napi_object) { type_error(env, "pcm description must be an object"); return 0; }
  if (prop_string(env, obj, "format", s, sizeof s))
    for (int i = 0; i < 5; ++i) if (!strcmp(s, kPcmNames[i])) pi->format = i;
  if (pi->format < 0) { type_error(env, "format must be one of u8, s16, s24, s32, f32"); return 0; }
  pi->channels = prop_double(env, obj, "channels", &d) ? (int32_t)d : 1;
  pi->sample_rate = prop_double(env, obj, "sampleRate", &d) ? (int32_t)d : 0;
  bpf = pi->channels * sg_pcm_sample_bytes(pi->format);
  if (pi->channels < 1 || pi->channels > 32 || n_clips < 1 || n_bytes % ((size_t)bpf * (size_t)n_clips)) {
    type_error(env, "samples length is not clips x frames x channels x sample size");
    return 0;
  }
  pi->frames = (int64_t)(n_bytes / ((size_t)bpf * (size_t)n_clips));
  return 1;
}

/* pcmDecode(engine, samples: Uint8Array, pcm, nClips, mix: 0|1, out: Float32Array): interleaved samples ->
 * float32 planes [clip][plane][frame]; mix = the AnalyserNode's speakers down-mix to mono */
static napi_value js_pcm_decode(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *e, *bytes, *out;
  size_t n, n_out;
  int32_t n_clips;
  int32_t mix = 0;
  sg_pcm_info pi;
  int rc, planes;
  if (get_args(env, info, argv) < 6 || !get_external(env, argv[0], &e)) return type_error(env, "pcmDecode(engine, samples, pcm, nClips, mix, out)");
  if (!get_typed(env, argv[1], napi_uint8_array, &bytes, &n)) return type_error(env, "samples must be a Uint8Array");
  if (napi_get_value_int32(env, argv[3], &n_clips) != napi_ok) return type_error(env, "nClips must be an integer");
  if (!parse_pcm(env, argv[2], n, n_clips, &pi)) return undefined_of(env);
  if (napi_get_value_int32(env, argv[4], &mix) != napi_ok) return type_error(env, "mix must be 0 or 1");
  if (!get_typed(env, argv[5], napi_float32_array, &out, &n_out)) return type_error(env, "out must be a Float32Array");
  planes = mix ? 1 : pi.channels;
  if (n_out < (size_t)n_clips * (size_t)planes * (size_t)pi.frames) return type_error(env, "out is smaller than clips x planes x frames");
  rc = sg_pcm_ingest((sg_engine*)e, bytes, n_clips, &pi, mix ? SG_PCM_MONO_MIX : SG_PCM_PLANAR, (float*)out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* stftPcm(engine, samples: Uint8Array, pcm, nClips, mix, options, out): the frame path fed with interleaved PCM */
static napi_value js_stft_pcm(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *e, *bytes, *out;
  size_t n, n_out;
  int32_t n_clips;
  int32_t mix = 1;
  sg_pcm_info pi;
  sg_stft_config cfg;
  int64_t frames;
  int rc, planes;
  if (get_args(env, info, argv) < 7 || !get_external(env, argv[0], &e)) return type_error(env, "stftPcm(engine, samples, pcm, nClips, mix, options, out)");
  if (!get_typed(env, argv[1], napi_uint8_array, &bytes, &n)) return type_error(env, "samples must be a Uint8Array");
  if (napi_get_value_int32(env, argv[3], &n_clips) != napi_ok) return type_error(env, "nClips must be an integer");
  if (!parse_pcm(env, argv[2], n, n_clips, &pi)) return undefined_of(env);
  if (napi_get_value_int32(env, argv[4], &mix) != napi_ok) return type_error(env, "mix must be 0 or 1");
  if (!parse_config(env, argv[5], &cfg)) return undefined_of(env);
  frames = sg_stft_num_frames(&cfg, pi.frames);
  if (frames < 0) return throw_status(env, SG_ERR_INDEX_SIZE);
  planes = mix ? 1 : pi.channels;
  if (!get_typed(env, argv[6], sg_stft_elem_bytes(&cfg) == 1 ? napi_uint8_array : (cfg.output == SG_OUT_RGBA8 ? napi_uint32_array : napi_float32_array), &out, &n_out))
    return type_error(env, "out has the wrong element type for options.output");
  if (n_out < (size_t)n_clips * (size_t)planes * (size_t)frames * (size_t)(cfg.n_fft / 2)) return type_error(env, "out is smaller than clips x planes x frames x bins");
  rc = sg_stft_pcm((sg_engine*)e, bytes, n_clips, &pi, mix ? SG_PCM_MONO_MIX : SG_PCM_PLANAR, &cfg, out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* resampleNumFrames(frames, inRate, outRate) -> the length after resampling: ceil(frames*up/down); host only */
static napi_value js_resample_num_frames(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS], r;
  int64_t frames, n;
  int32_t in_rate, out_rate;
  if (get_args(env, info, argv) < 3 || napi_get_value_int64(env, argv[0], &frames) != napi_ok ||
      napi_get_value_int32(env, argv[1], &in_rate) != napi_ok || napi_get_value_int32(env, argv[2], &out_rate) != napi_ok)
    return type_error(env, "resampleNumFrames(frames, inRate, outRate)");
  n = sg_resample_num_frames(frames, in_rate, out_rate);
  if (n < 0) return throw_status(env, (int)n);
  napi_create_double(env, (double)n, &r);
  return r;
}

/* pcmDecodeResampled(engine, samples, pcm, nClips, mix, outRate, out: Float32Array): pcmDecode, resampled from
 * pcm.sampleRate to outRate (decodeAudioData in a context running at outRate); out [clip][plane][resampled frame] */
static napi_value js_pcm_decode_resampled(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *e, *bytes, *out;
  size_t n, n_out;
  int32_t n_clips, out_rate;
  int32_t mix = 0;
  sg_pcm_info pi;
  int64_t length;
  int rc, planes;
  if (get_args(env, info, argv) < 7 || !get_external(env, argv[0], &e))
    return type_error(env, "pcmDecodeResampled(engine, samples, pcm, nClips, mix, outRate, out)");
  if (!get_typed(env, argv[1], napi_uint8_array, &bytes, &n)) return type_error(env, "samples must be a Uint8Array");
  if (napi_get_value_int32(env, argv[3], &n_clips) != napi_ok) return type_error(env, "nClips must be an integer");
  if (!parse_pcm(env, argv[2], n, n_clips, &pi)) return undefined_of(env);
  if (napi_get_value_int32(env, argv[4], &mix) != napi_ok) return type_error(env, "mix must be 0 or 1");
  if (napi_get_value_int32(env, argv[5], &out_rate) != napi_ok) return type_error(env, "outRate must be an integer");
  length = sg_resample_num_frames(pi.frames, pi.sample_rate, out_rate);
  if (length < 0) return throw_status(env, (int)length);
  if (!get_typed(env, argv[6], napi_float32_array, &out, &n_out)) return type_error(env, "out must be a Float32Array");
  planes = mix ? 1 : pi.channels;
  if (n_out < (size_t)n_clips * (size_t)planes * (size_t)length) return type_error(env, "out is smaller than clips x planes x resampled frames");
  rc = sg_pcm_ingest_resampled((sg_engine*)e, bytes, n_clips, &pi, mix ? SG_PCM_MONO_MIX : SG_PCM_PLANAR, out_rate, (float*)out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* stftPcmResampled(engine, samples, pcm, nClips, mix, outRate, options, out): stftPcm with the planes resampled
 * from pcm.sampleRate to outRate before framing */
static napi_value js_stft_pcm_resampled(napi_env env, napi_callback_info info) {
  napi_value argv[MAX_ARGS];
  void *e, *bytes, *out;
  size_t n, n_out;
  int32_t n_clips, out_rate;
  int32_t mix = 1;
  sg_pcm_info pi;
  sg_stft_config cfg;
  int64_t length, frames;
  int rc, planes;
  if (get_args(env, info, argv) < 8 || !get_external(env, argv[0], &e))
    return type_error(env, "stftPcmResampled(engine, samples, pcm, nClips, mix, outRate, options, out)");
  if (!get_typed(env, argv[1], napi_uint8_array, &bytes, &n)) return type_error(env, "samples must be a Uint8Array");
  if (napi_get_value_int32(env, argv[3], &n_clips) != napi_ok) return type_error(env, "nClips must be an integer");
  if (!parse_pcm(env, argv[2], n, n_clips, &pi)) return undefined_of(env);
  if (napi_get_value_int32(env, argv[4], &mix) != napi_ok) return type_error(env, "mix must be 0 or 1");
  if (napi_get_value_int32(env, argv[5], &out_rate) != napi_ok) return type_error(env, "outRate must be an integer");
  if (!parse_config(env, argv[6], &cfg)) return undefined_of(env);
  length = sg_resample_num_frames(pi.frames, pi.sample_rate, out_rate);
  if (length < 0) return throw_status(env, (int)length);
  frames = sg_stft_num_frames(&cfg, length);
  if (frames < 0) return throw_status(env, SG_ERR_INDEX_SIZE);
  planes = mix ? 1 : pi.channels;
  if (!get_typed(env, argv[7], sg_stft_elem_bytes(&cfg) == 1 ? napi_uint8_array : (cfg.output == SG_OUT_RGBA8 ? napi_uint32_array : napi_float32_array), &out, &n_out))
    return type_error(env, "out has the wrong element type for options.output");
  if (n_out < (size_t)n_clips * (size_t)planes * (size_t)frames * (size_t)(cfg.n_fft / 2)) return type_error(env, "out is smaller than clips x planes x frames x bins");
  rc = sg_stft_pcm_resampled((sg_engine*)e, bytes, n_clips, &pi, mix ? SG_PCM_MONO_MIX : SG_PCM_PLANAR, out_rate, &cfg, out);
  if (rc != SG_OK) return throw_status(env, rc);
  return undefined_of(env);
}

/* ---------------------------------------------------------------- module init */
static void export_fn(napi_env env, napi_value exports, const char* name, napi_callback cb) {
  napi_value fn;
  napi_create_function(env, name, NAPI_AUTO_LENGTH, cb, NULL, &fn);
  napi_set_named_property(env, exports, name, fn);
}

/* the only symbol Node looks up in an addon (what NAPI_MODULE_INIT() expands to) */
napi_value napi_register_module_v1(napi_env env, napi_value exports) {
  export_fn(env, exports, "deviceCount", js_device_count);
  export_fn(env, exports, "engineCreate", js_engine_create);
  export_fn(env, exports, "engineDestroy", js_engine_destroy);
  export_fn(env, exports, "engineLastKernel", js_engine_last_kernel);
  export_fn(env, exports, "numFrames", js_num_frames);
  export_fn(env, exports, "stftBatch", js_stft_batch);
  export_fn(env, exports, "stftBatchMulti", js_stft_batch_multi);
  export_fn(env, exports, "colormapReference", js_colormap_reference);
  export_fn(env, exports, "analyserCreate", js_analyser_create);
  export_fn(env, exports, "analyserDestroy", js_analyser_destroy);
  export_fn(env, exports, "analyserSet", js_analyser_set);
  export_fn(env, exports, "analyserGet", js_analyser_get);
  export_fn(env, exports, "analyserPush", js_analyser_push);
  export_fn(env, exports, "getByteFrequencyData", js_get_byte_frequency_data);
  export_fn(env, exports, "getFloatFrequencyData", js_get_float_frequency_data);
  export_fn(env, exports, "getByteTimeDomainData", js_get_byte_time_domain_data);
  export_fn(env, exports, "getFloatTimeDomainData", js_get_float_time_domain_data);
  export_fn(env, exports, "streamCreate", js_stream_create);
  export_fn(env, exports, "streamPush", js_stream_push);
  export_fn(env, exports, "streamDestroy", js_stream_destroy);
  export_fn(env, exports, "streamSetHistory", js_stream_set_history);
  export_fn(env, exports, "streamHistoryInfo", js_stream_history_info);
  export_fn(env, exports, "streamHistoryRead", js_stream_history_read);
  export_fn(env, exports, "streamView", js_stream_view);
  export_fn(env, exports, "ringCreate", js_ring_create);
  export_fn(env, exports, "ringAppend", js_ring_append);
  export_fn(env, exports, "ringYoffset", js_ring_yoffset);
  export_fn(env, exports, "ringView", js_ring_view);
  export_fn(env, exports, "ringDestroy", js_ring_destroy);
  export_fn(env, exports, "wavParse", js_wav_parse);
  export_fn(env, exports, "pcmDecode", js_pcm_decode);
  export_fn(env, exports, "stftPcm", js_stft_pcm);
  export_fn(env, exports, "resampleNumFrames", js_resample_num_frames);
  export_fn(env, exports, "pcmDecodeResampled", js_pcm_decode_resampled);
  export_fn(env, exports, "stftPcmResampled", js_stft_pcm_resampled);
  export_fn(env, exports, "biquadCoefficients", js_biquad_coefficients);
  export_fn(env, exports, "biquadFilter", js_biquad_filter);
  export_fn(env, exports, "streamSetFilter", js_stream_set_filter);
  return exports;
}

int32_t node_api_module_get_api_version_v1(void) { return 8; }
