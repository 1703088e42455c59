/* streams_smoke.c -- a plain C consumer of the per-stream calls of include/crispy_ns.h (subset calls, per-stream reset,
 * save / load of single streams), linked against libcrispy_ns.so.
 * A host subset call over streams {2, 0} of a batch of 4 must give each stream what a batch of its own gives; a stream
 * record moved into another slot continues it; a reset slot starts afresh.  Without a CUDA device it checks the
 * argument rules that need no handle and exits 0.
 * Build: gcc -std=c99 -Wall -Wextra -Werror -pedantic -Iinclude tests/c_abi/streams_smoke.c -Lcrispy_b200 -lcrispy_ns -lm
 */
#include "crispy_ns.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define CHECK(expr)                                                                                            \
  do {                                                                                                         \
    int rc_ = (expr);                                                                                          \
    if (rc_ != CRISPY_NS_OK) {                                                                                 \
      fprintf(stderr, "FAIL %s:%d: %s -> %d (%s)\n", __FILE__, __LINE__, #expr, rc_, crispy_ns_last_error()); \
      return 1;                                                                                                \
    }                                                                                                          \
  } while (0)
#define EXPECT(cond)                                                  \
  do {                                                                \
    if (!(cond)) {                                                    \
      fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); \
      return 1;                                                       \
    }                                                                 \
  } while (0)

enum { NF = 20, N = NF * CRISPY_NS_FRAME_SIZE };

static void make_signal(float *x, int n, unsigned seed) {
  unsigned r = seed * 2654435761u + 12345u;
  int i;
  for (i = 0; i < n; i++) {
    r = r * 1664525u + 1013904223u;
    x[i] = (float)(0.3 * sin(0.01 * i * (1 + seed)) + 0.05 * (((int)(r >> 16) & 0xFFFF) / 32768.0 - 1.0));
  }
}

/* one stream fed alone to a fresh batch of its own */
static int alone(const crispy_ns_model *m, const float *x, int n_frames, float *out, float *vad) {
  crispy_ns_batch *b = NULL;
  const int n = n_frames * CRISPY_NS_FRAME_SIZE;
  CHECK(crispy_ns_batch_create(m, 0, 1, &b));
  CHECK(crispy_ns_process_streams_host(b, x, out, vad, NULL, n_frames, n, n, n_frames, 0, CRISPY_NS_UNIT_SCALE, 1.0f));
  crispy_ns_batch_destroy(b);
  return 0;
}

int main(void) {
  crispy_ns_model *model = NULL;
  crispy_ns_batch *batch = NULL;
  const int ids[2] = {2, 0}, dup[2] = {1, 1};
  const size_t rec = crispy_ns_stream_state_size();
  static float x[2][N], out[2][N], vad[2][NF], want[N], wvad[NF];
  unsigned char *blob;
  int s, i;

  EXPECT(rec == 16 + 2784 * sizeof(float));
  EXPECT(crispy_ns_process_streams_subset(NULL, ids, 2, x, out, NULL, NULL, NF, N, N, 0, 0, 0, 1.0f, NULL) ==
         CRISPY_NS_EINVAL);
  EXPECT(crispy_ns_batch_reset_streams(NULL, ids, 2, NULL) == CRISPY_NS_EINVAL);
  EXPECT(crispy_ns_batch_save_streams(NULL, ids, 2, NULL, 0) == CRISPY_NS_EINVAL);
  EXPECT(crispy_ns_batch_load_streams(NULL, ids, 2, NULL, 0) == CRISPY_NS_EINVAL);
  if (crispy_ns_device_count() == 0) {
    printf("streams_smoke: no CUDA device, argument checks ok\n");
    return 0;
  }
  CHECK(crispy_ns_model_synthetic(0, &model));
  CHECK(crispy_ns_batch_create(model, 0, 4, &batch));
  EXPECT(crispy_ns_process_streams_subset_host(batch, dup, 2, x, out, NULL, NULL, NF, N, N, 0, 0, 0, 1.0f) ==
         CRISPY_NS_EINVAL);
  for (s = 0; s < 2; s++) make_signal(x[s], N, (unsigned)s + 1);
  CHECK(crispy_ns_process_streams_subset_host(batch, ids, 2, x, out, &vad[0][0], NULL, NF, N, N, NF, 0,
                                              CRISPY_NS_UNIT_SCALE, 1.0f));
  for (s = 0; s < 2; s++) {
    if (alone(model, x[s], NF, want, wvad)) return 1;
    EXPECT(memcmp(want, out[s], sizeof(want)) == 0);
    EXPECT(memcmp(wvad, vad[s], sizeof(wvad)) == 0);
  }
  {
    /* stream 2 (row 0) moves to slot 3 and continues there: its second half equals the uninterrupted run */
    const int from = 2, to = 3, half = NF / 2;
    float whole[N];
    blob = (unsigned char *)malloc(rec);
    EXPECT(blob != NULL);
    CHECK(crispy_ns_batch_reset_streams(batch, &from, 1, NULL));
    CHECK(crispy_ns_process_streams_subset_host(batch, &from, 1, x[0], out[0], NULL, NULL, half, N, N, 0, 0,
                                                CRISPY_NS_UNIT_SCALE, 1.0f));
    CHECK(crispy_ns_batch_save_streams(batch, &from, 1, blob, rec));
    EXPECT(memcmp(blob, "CRNSSTR1", 8) == 0);
    CHECK(crispy_ns_batch_load_streams(batch, &to, 1, blob, rec));
    EXPECT(crispy_ns_batch_load_streams(batch, &to, 1, blob, rec - 1) == CRISPY_NS_EINVAL);
    CHECK(crispy_ns_process_streams_subset_host(batch, &to, 1, x[0] + half * CRISPY_NS_FRAME_SIZE, out[1], NULL, NULL,
                                                NF - half, N, N, 0, 0, CRISPY_NS_UNIT_SCALE, 1.0f));
    if (alone(model, x[0], NF, whole, wvad)) return 1;
    for (i = 0; i < (NF - half) * CRISPY_NS_FRAME_SIZE; i++) EXPECT(out[1][i] == whole[half * CRISPY_NS_FRAME_SIZE + i]);
    free(blob);
  }
  crispy_ns_batch_destroy(batch);
  crispy_ns_model_destroy(model);
  printf("streams_smoke: ok\n");
  return 0;
}
