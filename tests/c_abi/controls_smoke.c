/* controls_smoke.c -- a plain C consumer of the per-stream suppression controls of include/crispy_ns.h
 * (crispy_ns_controls: attenuation limit and voice gate), linked against libcrispy_ns.so.
 * In a batch of 3, stream 1 gets a gate that never opens (threshold 1, hold 0, gate gain 0): its first frame ramps
 * down to silence and every later frame is exactly zero, while streams 0 and 2 give what a batch without controls
 * gives.  get_controls reads back what set_controls stored, a bad value changes nothing, and a per-stream reset turns
 * the controls off.  Without a CUDA device it checks the argument rules that need no handle and exits 0.
 * Build: gcc -std=c99 -Wall -Wextra -Werror -pedantic -Iinclude tests/c_abi/controls_smoke.c -Lcrispy_b200 -lcrispy_ns -lm
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

enum { NS = 3, NF = 12, N = NF * CRISPY_NS_FRAME_SIZE };

static void make_signal(float *x, int n, unsigned seed) {
  unsigned r = seed * 2654435761u + 12345u;
  int i;
  for (i = 0; i < n; i++) {
    r = r * 1664525u + 1013904223u;
    x[i] = (float)(0.3 * sin(0.01 * i * (1 + seed)) + 0.05 * (((int)(r >> 16) & 0xFFFF) / 32768.0 - 1.0));
  }
}

static int same_controls(const crispy_ns_controls *a, const crispy_ns_controls *b) {
  return a->min_gain == b->min_gain && a->gate_threshold == b->gate_threshold && a->gate_hold == b->gate_hold &&
         a->gate_gain == b->gate_gain;
}

int main(void) {
  static float in[NS * N], out[NS * N], ref[NS * N], vad[NS * NF];
  const crispy_ns_controls off = {0.f, 0.f, 0, 0.f};
  const crispy_ns_controls closed = {0.f, 1.f, 0, 0.f};
  crispy_ns_controls bad = closed, got[NS];
  crispy_ns_batch *b = NULL, *plain = NULL;
  crispy_ns_state *st = NULL;
  int ids[NS] = {0, 1, 2}, one = 1, i, s, rc;
  EXPECT(crispy_ns_batch_set_controls(NULL, &one, 1, &closed, NULL) == CRISPY_NS_EINVAL);
  EXPECT(crispy_ns_batch_get_controls(NULL, &one, 1, got) == CRISPY_NS_EINVAL);
  EXPECT(crispy_ns_set_controls(NULL, &closed) == CRISPY_NS_EINVAL);
  EXPECT(crispy_ns_get_controls(NULL, got) == CRISPY_NS_EINVAL);
  EXPECT(crispy_ns_multi_set_controls(NULL, &one, 1, &closed) == CRISPY_NS_EINVAL);
  EXPECT(crispy_ns_multi_get_controls(NULL, &one, 1, got) == CRISPY_NS_EINVAL);
  rc = crispy_ns_batch_create(NULL, 0, NS, &b);
  if (crispy_ns_device_count() == 0) {
    EXPECT(rc == CRISPY_NS_ENODEV && b == NULL);
    EXPECT(crispy_ns_create(NULL, 0, &st) == CRISPY_NS_ENODEV);
    printf("controls_smoke: ENODEV contract ok\n");
    return 0;
  }
  CHECK(rc);
  CHECK(crispy_ns_batch_create(NULL, 0, NS, &plain));
  for (s = 0; s < NS; s++) make_signal(in + (size_t)s * N, N, (unsigned)s + 7u);

  CHECK(crispy_ns_batch_get_controls(b, ids, NS, got));
  for (s = 0; s < NS; s++) EXPECT(same_controls(&got[s], &off));
  CHECK(crispy_ns_batch_set_controls(b, &one, 1, &closed, NULL));
  bad.gate_gain = NAN;
  EXPECT(crispy_ns_batch_set_controls(b, &one, 1, &bad, NULL) == CRISPY_NS_EINVAL);
  bad = closed;
  bad.gate_hold = (1 << 20) + 1;
  EXPECT(crispy_ns_batch_set_controls(b, &one, 1, &bad, NULL) == CRISPY_NS_EINVAL);
  CHECK(crispy_ns_batch_get_controls(b, &one, 1, got));
  EXPECT(same_controls(&got[0], &closed));

  CHECK(crispy_ns_process_streams_host(b, in, out, vad, NULL, NF, N, N, NF, 0, CRISPY_NS_UNIT_SCALE, 1.0f));
  CHECK(crispy_ns_process_streams_host(plain, in, ref, NULL, NULL, NF, N, N, 0, 0, CRISPY_NS_UNIT_SCALE, 1.0f));
  EXPECT(memcmp(out, ref, sizeof(float) * N) == 0);
  EXPECT(memcmp(out + 2 * N, ref + 2 * N, sizeof(float) * N) == 0);
  for (i = 0; i < CRISPY_NS_FRAME_SIZE; i++) { /* frame 0: G ramps from 1 down to 0 */
    const float gr = 1.f + (0.f - 1.f) * ((float)(i + 1) / 480.0f);
    const float want = fminf(1.f, fmaxf(-1.f, (ref[N + i] * 32768.0f * gr) / 32768.0f));
    EXPECT(fabsf(out[N + i] - want) <= 1e-6f);
  }
  for (i = CRISPY_NS_FRAME_SIZE; i < N; i++) EXPECT(out[N + i] == 0.f);

  CHECK(crispy_ns_batch_reset_streams(b, &one, 1, NULL));
  CHECK(crispy_ns_batch_get_controls(b, &one, 1, got));
  EXPECT(same_controls(&got[0], &off));

  CHECK(crispy_ns_create(NULL, 0, &st));
  CHECK(crispy_ns_set_controls(st, &closed));
  CHECK(crispy_ns_get_controls(st, got));
  EXPECT(same_controls(&got[0], &closed));
  CHECK(crispy_ns_reset(st));
  CHECK(crispy_ns_get_controls(st, got));
  EXPECT(same_controls(&got[0], &off));
  crispy_ns_destroy(st);
  crispy_ns_batch_destroy(plain);
  crispy_ns_batch_destroy(b);
  printf("controls_smoke: ok\n");
  return 0;
}
