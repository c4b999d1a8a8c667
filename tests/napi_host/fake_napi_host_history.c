/*
 * fake_napi_host_history.c -- the sonogram-history natives of spectrogram.node (streamSetHistory, streamHistoryInfo,
 * streamHistoryRead, streamView, and streamPush without an out array) driven through the fake Node runtime of
 * fake_napi_host.c (its value model, call/expect helpers and driver are reused as they are; only its main is renamed).
 * Test infrastructure only.
 *
 *   fake_napi_host_history <spectrogram.node> cpu            exports and handle checks (no device needed)
 *   fake_napi_host_history <spectrogram.node> gpu <out.bin>  a history-enabled bank on device 0: argument checks, then
 *                                                            the texture and two views written to out.bin
 */
#define main fake_napi_host_main
#include "fake_napi_host.c"
#undef main

enum { H_CH = 8, H_BINS = 512, H_ROWS = 24, H_MAX_CHUNK = 1024 };

/* uniform samples in [-0.5, 0.5) from a 32-bit LCG, exact in float32 (reproduced by tests/test_stream_history.py) */
static uint32_t g_lcg = 2024u;
static float next_sample(void) {
  g_lcg = g_lcg * 1664525u + 1013904223u;
  return (float)((double)(g_lcg >> 8) / 16777216.0 - 0.5);
}

static void history_cpu_checks(void) {
  const char* names[] = {"streamSetHistory", "streamHistoryInfo", "streamHistoryRead", "streamView", "streamPush"};
  for (size_t i = 0; i < sizeof names / sizeof *names; ++i) {
    prop* p = find_prop(g_exports, names[i]);
    expect(p && p->value->type == napi_function, names[i]);
  }
  uint32_t img[16];
  unsigned char tex[16];
  napi_value a[6];
  a[0] = num(7); a[1] = num(16);
  call("streamSetHistory", 2, a);
  expect(threw("TypeError", NULL), "streamSetHistory(non-stream) -> TypeError");
  call("streamHistoryInfo", 1, a);
  expect(threw("TypeError", NULL), "streamHistoryInfo(non-stream) -> TypeError");
  a[1] = num(0); a[2] = num(1); a[3] = typed(napi_uint8_array, 16, tex);
  call("streamHistoryRead", 4, a);
  expect(threw("TypeError", NULL), "streamHistoryRead(non-stream) -> TypeError");
  a[3] = num(2); a[4] = num(2); a[5] = typed(napi_uint32_array, 16, img);
  call("streamView", 6, a);
  expect(threw("TypeError", NULL), "streamView(non-stream) -> TypeError");
  call("streamView", 5, a);
  expect(threw("TypeError", NULL), "streamView with five arguments -> TypeError");
}

static void history_gpu_run(const char* out_path) {
  const int chunks[] = {256, 1024, 128, 1024, 1024, 512, 1024, 1024};   /* 47 frames: the 24-row texture wraps */
  const size_t n_tex = (size_t)H_CH * H_ROWS * H_BINS, n_v1 = (size_t)H_CH * 32 * 64, n_v2 = (size_t)3 * 7 * 33;
  float* chunk = (float*)malloc(sizeof(float) * H_CH * H_MAX_CHUNK);
  unsigned char* rows = (unsigned char*)malloc((size_t)H_CH * (H_MAX_CHUNK / 128) * H_BINS);
  unsigned char* tex = (unsigned char*)calloc(n_tex, 1);
  uint32_t *v1 = (uint32_t*)calloc(n_v1, 4), *v2 = (uint32_t*)calloc(n_v2, 4);
  napi_value a[6], r;
  a[0] = num(0);
  napi_value eng = call("engineCreate", 1, a);
  expect(!g_env.pending && eng->type == napi_external, "engineCreate(0)");
  a[0] = eng; a[1] = num(H_CH); a[2] = options(1024, 128, "u8", NULL); a[3] = num(H_MAX_CHUNK);
  napi_value st = call("streamCreate", 4, a);
  expect(!g_env.pending && st->type == napi_external, "streamCreate(8 channels, n_fft 1024, hop 128)");
  a[0] = st;
  r = call("streamHistoryInfo", 1, a);
  expect(!g_env.pending && find_prop(r, "rows")->value->num == 0, "streamHistoryInfo: rows 0 before a history is attached");
  a[1] = num(0); a[2] = num(H_CH); a[3] = num(64); a[4] = num(32); a[5] = typed(napi_uint32_array, n_v1, v1);
  call("streamView", 6, a);
  expect(threw("Error", "InvalidStateError"), "streamView without a history -> Error[InvalidStateError]");
  a[1] = typed(napi_float32_array, (size_t)H_CH * 128, chunk); a[2] = num(128); a[3] = new_value(napi_undefined);
  call("streamPush", 4, a);
  expect(threw("TypeError", NULL), "streamPush with an undefined out and no history -> TypeError");
  a[1] = num(1);
  call("streamSetHistory", 2, a);
  expect(threw("TypeError", NULL), "streamSetHistory(1 row) -> TypeError");
  a[1] = num(H_ROWS);
  call("streamSetHistory", 2, a);
  expect(!g_env.pending, "streamSetHistory(24 rows)");
  for (size_t k = 0; k < sizeof chunks / sizeof *chunks; ++k) {
    const int len = chunks[k];
    for (int i = 0; i < H_CH * len; ++i) chunk[i] = next_sample();
    a[0] = st; a[1] = typed(napi_float32_array, (size_t)H_CH * len, chunk); a[2] = num(len);
    a[3] = k % 2 ? new_value(napi_undefined) : typed(napi_uint8_array, (size_t)H_CH * (len / 128) * H_BINS, rows);
    call("streamPush", 4, a);
    expect(!g_env.pending, k % 2 ? "streamPush(out undefined): rows only reach the history" : "streamPush(out)");
  }
  a[3] = new_value(napi_undefined); a[4] = typed(napi_uint32_array, (size_t)H_CH * 8 * H_BINS, v1);
  call("streamPush", 5, a);
  expect(threw("TypeError", NULL), "streamPush with outRgba but no out -> TypeError");
  a[0] = st;
  r = call("streamHistoryInfo", 1, a);
  expect(!g_env.pending && find_prop(r, "rows")->value->num == H_ROWS && find_prop(r, "yoffset")->value->num == 47 % H_ROWS,
         "streamHistoryInfo: {rows 24, yoffset 47 % 24}");
  a[1] = num(0); a[2] = num(H_CH); a[3] = typed(napi_uint8_array, n_tex, tex);
  call("streamHistoryRead", 4, a);
  expect(!g_env.pending, "streamHistoryRead(all channels)");
  a[3] = typed(napi_uint8_array, n_tex - 1, tex);
  call("streamHistoryRead", 4, a);
  expect(threw("TypeError", NULL), "streamHistoryRead with a short out -> TypeError");
  a[1] = num(0); a[2] = num(H_CH); a[3] = num(64); a[4] = num(32); a[5] = typed(napi_uint32_array, n_v1, v1);
  call("streamView", 6, a);
  expect(!g_env.pending, "streamView(all channels, 64 x 32)");
  a[1] = num(2); a[2] = num(3); a[3] = num(33); a[4] = num(7); a[5] = typed(napi_uint32_array, n_v2, v2);
  call("streamView", 6, a);
  expect(!g_env.pending, "streamView(channels 2..4, 33 x 7)");
  a[5] = typed(napi_uint32_array, n_v2 - 1, v2);
  call("streamView", 6, a);
  expect(threw("TypeError", NULL), "streamView with a short out -> TypeError");
  a[5] = typed(napi_uint8_array, n_v2 * 4, v2);
  call("streamView", 6, a);
  expect(threw("TypeError", NULL), "streamView with a Uint8Array out -> TypeError");
  a[5] = typed(napi_uint32_array, n_v2, v2);
  a[1] = num(6);
  call("streamView", 6, a);
  expect(threw("TypeError", NULL), "streamView of channels 6..8 of 8 -> TypeError");
  a[1] = num(-1);
  call("streamView", 6, a);
  expect(threw("TypeError", NULL), "streamView from channel -1 -> TypeError");
  a[1] = num(0); a[2] = num(0);
  call("streamView", 6, a);
  expect(threw("TypeError", NULL), "streamView of 0 channels -> TypeError");
  a[2] = num(1); a[3] = num(0);
  call("streamView", 6, a);
  expect(threw("TypeError", NULL), "streamView 0 pixels wide -> TypeError");
  FILE* f = fopen(out_path, "wb");
  fwrite(tex, 1, n_tex, f);
  fwrite(v1, 4, n_v1, f);
  fwrite(v2, 4, n_v2, f);
  fclose(f);
  a[0] = st; a[1] = num(0);
  call("streamSetHistory", 2, a);
  expect(!g_env.pending, "streamSetHistory(0) detaches");
  a[1] = num(0); a[2] = num(1); a[3] = num(33); a[4] = num(7); a[5] = typed(napi_uint32_array, n_v2, v2);
  call("streamView", 6, a);
  expect(threw("Error", "InvalidStateError"), "streamView after detaching -> Error[InvalidStateError]");
  a[0] = st;
  call("streamDestroy", 1, a);
  a[0] = eng;
  call("engineDestroy", 1, a);
}

int main(int argc, char** argv) {
  if (argc < 3) { fprintf(stderr, "usage: %s spectrogram.node cpu|gpu [out.bin]\n", argv[0]); return 2; }
  void* h = dlopen(argv[1], RTLD_NOW | RTLD_GLOBAL);
  if (!h) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 2; }
  napi_value (*init)(napi_env, napi_value) = (napi_value(*)(napi_env, napi_value))dlsym(h, "napi_register_module_v1");
  if (!init) { fprintf(stderr, "addon does not export napi_register_module_v1\n"); return 2; }
  g_exports = new_value(napi_object);
  g_exports = init(&g_env, g_exports);
  history_cpu_checks();
  if (!strcmp(argv[2], "gpu")) history_gpu_run(argc > 3 ? argv[3] : "napi_history.bin");
  printf("%d failure(s)\n", g_failures);
  return g_failures ? 1 : 0;
}
