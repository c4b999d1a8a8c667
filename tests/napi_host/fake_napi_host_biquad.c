/*
 * fake_napi_host_biquad.c -- the biquad natives of spectrogram.node (biquadCoefficients, biquadFilter, streamSetFilter)
 * driven through the fake Node runtime of fake_napi_host.c (its value model, call/expect helpers and driver are reused
 * as they are; only its main is renamed).  Test infrastructure only.
 *
 *   fake_napi_host_biquad <spectrogram.node> cpu            exports, parameter and array-length checks (no device needed)
 *   fake_napi_host_biquad <spectrogram.node> gpu <out.bin>  on device 0: 3 channels filtered in two calls with the state
 *                                                           carried, then a 4-channel bank with a bandpass; the samples,
 *                                                           the state and the bank's byte rows written to out.bin
 */
#define main fake_napi_host_main
#include "fake_napi_host.c"
#undef main

/* uniform samples in [-0.5, 0.5) from a 32-bit LCG, exact in float32 (tests/test_stream_history.py lcg_chunks) */
static uint32_t g_lcg = 2024u;
static float next_sample(void) {
  g_lcg = g_lcg * 1664525u + 1013904223u;
  return (float)((double)(g_lcg >> 8) / 16777216.0 - 0.5);
}

static napi_value bq_params(const char* type, double frequency, double q) {
  napi_value o = new_value(napi_object);
  napi_set_named_property(&g_env, o, "type", str(type));
  napi_set_named_property(&g_env, o, "sampleRate", num(48000));
  napi_set_named_property(&g_env, o, "frequency", num(frequency));
  napi_set_named_property(&g_env, o, "Q", num(q));
  return o;
}

static void biquad_cpu_checks(void) {
  const char* names[] = {"biquadCoefficients", "biquadFilter", "streamSetFilter"};
  for (size_t i = 0; i < sizeof names / sizeof *names; ++i) {
    prop* p = find_prop(g_exports, names[i]);
    expect(p && p->value->type == napi_function, names[i]);
  }
  double coef[5] = {0}, st[12] = {0};
  float in[64] = {0}, out[64] = {0};
  int dummy = 0;
  napi_value a[7];
  a[0] = bq_params("bandpass", 1000, 10); a[1] = typed(napi_float64_array, 5, coef);
  call("biquadCoefficients", 2, a);
  expect(!g_env.pending && coef[1] == 0.0 && coef[0] > 0.0 && coef[2] == -coef[0], "biquadCoefficients(bandpass)");
  a[0] = bq_params("bogus", 1000, 10);
  call("biquadCoefficients", 2, a);
  expect(threw("TypeError", NULL), "biquadCoefficients(unknown type) -> TypeError");
  a[0] = bq_params("notch", NAN, 10);
  call("biquadCoefficients", 2, a);
  expect(threw("TypeError", NULL), "biquadCoefficients(frequency NaN) -> TypeError");
  a[0] = bq_params("notch", 1000, 10); a[1] = typed(napi_float64_array, 4, coef);
  call("biquadCoefficients", 2, a);
  expect(threw("TypeError", NULL), "biquadCoefficients with a 4-entry out -> TypeError");
  a[1] = typed(napi_float32_array, 5, in);
  call("biquadCoefficients", 2, a);
  expect(threw("TypeError", NULL), "biquadCoefficients with a Float32Array out -> TypeError");
  /* a stand-in engine handle: every one of these calls must fail its checks before the pointer reaches the core */
  a[0] = new_value(napi_external); a[0]->ext = &dummy;
  a[1] = bq_params("bandpass", 1000, 10); a[2] = typed(napi_float32_array, 64, in); a[3] = num(3); a[4] = num(22);
  a[5] = typed(napi_float64_array, 12, st); a[6] = typed(napi_float32_array, 64, out);
  call("biquadFilter", 7, a);
  expect(threw("TypeError", NULL), "biquadFilter with 64 samples for 3 x 22 -> TypeError");
  a[4] = num(21); a[6] = typed(napi_float32_array, 62, out);
  call("biquadFilter", 7, a);
  expect(threw("TypeError", NULL), "biquadFilter with 62 outputs for 3 x 21 -> TypeError");
  a[6] = typed(napi_float32_array, 64, out); a[5] = typed(napi_float64_array, 11, st);
  call("biquadFilter", 7, a);
  expect(threw("TypeError", NULL), "biquadFilter with 11 state values for 3 channels -> TypeError");
  a[5] = typed(napi_float32_array, 12, in);
  call("biquadFilter", 7, a);
  expect(threw("TypeError", NULL), "biquadFilter with a Float32Array state -> TypeError");
  a[5] = typed(napi_float64_array, 12, st); a[3] = num(-1);
  call("biquadFilter", 7, a);
  expect(threw("TypeError", NULL), "biquadFilter with -1 channels -> TypeError");
  a[3] = num(3); a[1] = bq_params("bogus", 1000, 10);
  call("biquadFilter", 7, a);
  expect(threw("TypeError", NULL), "biquadFilter(unknown type) -> TypeError");
  a[0] = num(7); a[1] = bq_params("bandpass", 1000, 10);
  call("streamSetFilter", 2, a);
  expect(threw("TypeError", NULL), "streamSetFilter(non-stream) -> TypeError");
}

static void biquad_gpu_run(const char* out_path) {
  enum { CH = 3, L0 = 5000, L1 = 3000, BCH = 4 };
  const int lens[2] = {L0, L1}, pushes[3] = {1024, 512, 1024};
  float* x = (float*)malloc(sizeof(float) * CH * L0);
  float* yc = (float*)malloc(sizeof(float) * CH * L0);
  float* y = (float*)malloc(sizeof(float) * CH * (L0 + L1));
  unsigned char* rows = (unsigned char*)malloc((size_t)BCH * 8 * 512);
  double st[CH * 4] = {0};
  napi_value a[7];
  a[0] = num(0);
  napi_value eng = call("engineCreate", 1, a);
  expect(!g_env.pending && eng->type == napi_external, "engineCreate(0)");
  FILE* f = fopen(out_path, "wb");
  for (int k = 0, off = 0; k < 2; off += lens[k], ++k) {
    for (int i = 0; i < CH * lens[k]; ++i) x[i] = next_sample();
    a[0] = eng; a[1] = bq_params("bandpass", 1200, 10); a[2] = typed(napi_float32_array, (size_t)CH * lens[k], x);
    a[3] = num(CH); a[4] = num(lens[k]); a[5] = typed(napi_float64_array, CH * 4, st);
    a[6] = typed(napi_float32_array, (size_t)CH * lens[k], yc);
    call("biquadFilter", 7, a);
    expect(!g_env.pending, "biquadFilter(3 channels, state carried)");
    for (int c = 0; c < CH; ++c) memcpy(y + (size_t)c * (L0 + L1) + off, yc + (size_t)c * lens[k], sizeof(float) * lens[k]);
  }
  fwrite(y, sizeof(float), (size_t)CH * (L0 + L1), f);
  fwrite(st, sizeof(double), CH * 4, f);
  a[0] = eng; a[1] = num(BCH); a[2] = options(1024, 128, "u8", NULL); a[3] = num(1024);
  napi_value s = call("streamCreate", 4, a);
  expect(!g_env.pending && s->type == napi_external, "streamCreate(4 channels)");
  a[0] = s; a[1] = bq_params("bogus", 2500, 10);
  call("streamSetFilter", 2, a);
  expect(threw("TypeError", NULL), "streamSetFilter(unknown type) -> TypeError");
  a[1] = bq_params("bandpass", 2500, 10);
  call("streamSetFilter", 2, a);
  expect(!g_env.pending, "streamSetFilter(bandpass)");
  g_lcg = 77u;
  for (int k = 0; k < 3; ++k) {
    for (int i = 0; i < BCH * pushes[k]; ++i) x[i] = next_sample();
    const size_t n_rows = (size_t)BCH * (pushes[k] / 128) * 512;
    a[0] = s; a[1] = typed(napi_float32_array, (size_t)BCH * pushes[k], x); a[2] = num(pushes[k]);
    a[3] = typed(napi_uint8_array, n_rows, rows);
    call("streamPush", 4, a);
    expect(!g_env.pending, "streamPush through the filter");
    fwrite(rows, 1, n_rows, f);
  }
  fclose(f);
  a[0] = s; a[1] = new_value(napi_null);
  call("streamSetFilter", 2, a);
  expect(!g_env.pending, "streamSetFilter(null) detaches");
  call("streamDestroy", 1, a);
  a[0] = eng;
  call("engineDestroy", 1, a);
  free(x); free(yc); free(y); free(rows);
}

int main(int argc, char** argv) {
  if (argc < 3) { fprintf(stderr, "usage: %s spectrogram.node cpu|gpu [out.bin]\n", argv[0]); return 2; }
  void* h = dlopen(argv[1], RTLD_NOW | RTLD_GLOBAL);
  if (!h) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 2; }
  napi_value (*init)(napi_env, napi_value) = (napi_value(*)(napi_env, napi_value))dlsym(h, "napi_register_module_v1");
  if (!init) { fprintf(stderr, "addon does not export napi_register_module_v1\n"); return 2; }
  g_exports = new_value(napi_object);
  g_exports = init(&g_env, g_exports);
  biquad_cpu_checks();
  if (!strcmp(argv[2], "gpu")) biquad_gpu_run(argc > 3 ? argv[3] : "napi_biquad.bin");
  printf("%d failure(s)\n", g_failures);
  return g_failures ? 1 : 0;
}
