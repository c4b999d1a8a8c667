/*
 * fake_napi_host_resample.c -- the resampling natives of spectrogram.node driven through the fake Node runtime of
 * fake_napi_host.c (its value model, call/expect helpers and driver are reused as they are; only its main is renamed).
 * Test infrastructure only.
 *
 *   fake_napi_host_resample <spectrogram.node> <out.bin>  boundary checks of the resampling natives, then a run on
 *                                                         device 0 writing the resampled planes and spectrogram bytes
 */
#define main fake_napi_host_main
#include "fake_napi_host.c"
#undef main

/* 1 s of s16 stereo at 44.1 kHz (a 32-bit LCG, reproducible in Python), resampled to 48 kHz: mono-mix planes from
 * pcmDecodeResampled, then stftPcmResampled bytes (n_fft 2048, hop 512, u8), both written to out_path */
static void resample_run(const char* out_path) {
  napi_value a[8], r, desc = new_value(napi_object);
  const int n = 44100, len = 48000, frames = 1 + (len - 2048) / 512, bins = 1024;
  short* s16 = (short*)malloc(sizeof(short) * 2 * n);
  float* dec = (float*)calloc(len, sizeof(float));
  unsigned char* spec = (unsigned char*)calloc((size_t)frames * bins, 1);
  uint32_t state = 12345u;
  for (int i = 0; i < 2 * n; ++i) { state = state * 1664525u + 1013904223u; s16[i] = (short)(state >> 16); }
  a[0] = num(n); a[1] = num(44100); a[2] = num(48000);
  r = call("resampleNumFrames", 3, a);
  expect(!g_env.pending && r->num == len, "resampleNumFrames(44100, 44100, 48000) == 48000");
  a[2] = num(48001);
  call("resampleNumFrames", 3, a);
  expect(threw("RangeError", "IndexSizeError"), "resampleNumFrames(.., 44100, 48001): ratio too fine -> IndexSizeError");
  a[0] = num(0);
  napi_value eng = call("engineCreate", 1, a);
  expect(!g_env.pending && eng->type == napi_external, "engineCreate(0)");
  napi_set_named_property(&g_env, desc, "format", str("s16"));
  napi_set_named_property(&g_env, desc, "channels", num(2));
  napi_set_named_property(&g_env, desc, "sampleRate", num(44100));
  a[0] = eng; a[1] = typed(napi_uint8_array, sizeof(short) * 2 * n, s16); a[2] = desc; a[3] = num(1); a[4] = num(1);
  a[5] = num(48000); a[6] = typed(napi_float32_array, len, dec);
  call("pcmDecodeResampled", 7, a);
  expect(!g_env.pending, "pcmDecodeResampled(s16 stereo 44.1 kHz, mix, 48 kHz)");
  a[6] = typed(napi_float32_array, len - 1, dec);
  call("pcmDecodeResampled", 7, a);
  expect(threw("TypeError", NULL), "pcmDecodeResampled with a short out -> TypeError");
  a[5] = num(2000); a[6] = typed(napi_float32_array, len, dec);
  call("pcmDecodeResampled", 7, a);
  expect(threw("RangeError", "IndexSizeError"), "pcmDecodeResampled to 2000 Hz -> IndexSizeError");
  a[5] = num(48000); a[6] = options(2048, 512, "u8", "valid"); a[7] = typed(napi_uint8_array, (size_t)frames * bins, spec);
  call("stftPcmResampled", 8, a);
  expect(!g_env.pending, "stftPcmResampled(s16 stereo 44.1 kHz, mix, 48 kHz)");
  a[7] = typed(napi_uint8_array, (size_t)frames * bins - 1, spec);
  call("stftPcmResampled", 8, a);
  expect(threw("TypeError", NULL), "stftPcmResampled with a short out -> TypeError");
  FILE* f = fopen(out_path, "wb");
  fwrite(dec, sizeof(float), len, f);
  fwrite(spec, 1, (size_t)frames * bins, f);
  fclose(f);
  a[0] = eng;
  call("engineDestroy", 1, a);
}

int main(int argc, char** argv) {
  if (argc < 3) { fprintf(stderr, "usage: %s spectrogram.node out.bin\n", argv[0]); return 2; }
  void* h = dlopen(argv[1], RTLD_NOW | RTLD_GLOBAL);
  if (!h) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 2; }
  napi_value (*init)(napi_env, napi_value) = (napi_value(*)(napi_env, napi_value))dlsym(h, "napi_register_module_v1");
  if (!init) { fprintf(stderr, "addon does not export napi_register_module_v1\n"); return 2; }
  g_exports = new_value(napi_object);
  g_exports = init(&g_env, g_exports);
  const char* names[] = {"resampleNumFrames", "pcmDecodeResampled", "stftPcmResampled"};
  for (size_t i = 0; i < sizeof names / sizeof *names; ++i) {
    prop* p = find_prop(g_exports, names[i]);
    expect(p && p->value->type == napi_function, names[i]);
  }
  resample_run(argv[2]);
  printf("%d failure(s)\n", g_failures);
  return g_failures ? 1 : 0;
}
