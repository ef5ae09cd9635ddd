/* oracle/restate/dnn.c -- TEST INFRASTRUCTURE (CPU restatement, see oracle.h).
 *
 * DNN-HMM forward exactly as the reference's x86 FMA path computes it:
 *   logistic table + clamp      libsent/src/phmm/calc_dnn.c:342-369
 *   calc_dnn_fma (GEMV)         libsent/src/phmm/calc_dnn_fma.c:18-95  (8 partial sums by lane,
 *                               horizontal add in lane order, + bias); scalar sub1 (calc_dnn.c:509-523)
 *                               when the input length is not a multiple of 8.  The reference itself is no
 *                               guide there: its FMA GEMV runs over in/8 blocks and drops the rest (its AVX
 *                               and SSE variants refuse such layers, calc_dnn.c:395-401), so this path is
 *                               held against float64 instead (tests/test_scoring_reference.py)
 *   dnn_calc_outprob            libsent/src/phmm/calc_dnn.c:774-868    (hidden: logistic table;
 *                               output: linear; log-softmax through addlog_array; * INV_LOG_TEN - prior)
 */
#include <math.h>
#include "oracle.h"

#define LOGISTIC_TABLE_FACTOR 20000
#define LOGISTIC_TABLE_MAX (16 * LOGISTIC_TABLE_FACTOR)
#define LOGISTIC_MIN 0.000334
#define LOGISTIC_MAX 0.999666

static float g_logistic[LOGISTIC_TABLE_MAX + 1];
static int g_logistic_built = 0;

void oracle_logistic_table(float *out) {
  int i;
  if (!g_logistic_built) {
    for (i = 0; i <= LOGISTIC_TABLE_MAX; i++) {
      double x = (double)i / (double)LOGISTIC_TABLE_FACTOR - 8.0;
      double d = 1.0 / (1.0 + exp(-x));
      g_logistic[i] = (float)d;
    }
    g_logistic_built = 1;
  }
  if (out) memcpy(out, g_logistic, sizeof(g_logistic));
}

static float logistic_func(float x) {
  if (x <= -8.0f) return LOGISTIC_MIN;
  if (x >= 8.0f) return LOGISTIC_MAX;
  return g_logistic[(int)((x + 8.0f) * LOGISTIC_TABLE_FACTOR + 0.5)];
}

static void gemv(float *dst, const float *src, const float *w, const float *b, int out, int in) {
  int i, j, l;
  if (in % 8 == 0) {
    int n = in / 8;
    for (i = 0; i < out; i++) {
      float x[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      const float *wr = w + (size_t)i * in;
      for (j = 0; j < n; j++)
        for (l = 0; l < 8; l++) x[l] = fmaf(src[8 * j + l], wr[8 * j + l], x[l]);
      dst[i] = x[0] + x[1] + x[2] + x[3] + x[4] + x[5] + x[6] + x[7] + b[i];
    }
  } else {
    for (i = 0; i < out; i++) {
      float x = 0.0f;
      const float *wr = w + (size_t)i * in;
      for (j = 0; j < in; j++) x += wr[j] * src[j];
      dst[i] = x + b[i];
    }
  }
}

int oracle_dnn_score(const jb200_dnn_desc *d, const float *in, int T, float *out) {
  int t, l, i, maxw = d->in_dim;
  float *bufa, *bufb;
  oracle_logistic_table(NULL);
  oracle_addlog_table(NULL);
  for (l = 0; l < d->n_layers; l++) if (d->layer_out[l] > maxw) maxw = d->layer_out[l];
  bufa = (float *)malloc(sizeof(float) * maxw);
  bufb = (float *)malloc(sizeof(float) * maxw);
  for (t = 0; t < T; t++) {
    const float *src = in + (size_t)t * d->in_dim;
    float *dst = bufa;
    float *row = out + (size_t)t * d->out_dim;
    float logprob;
    for (l = 0; l < d->n_layers - 1; l++) {
      gemv(dst, src, d->w[l], d->b[l], d->layer_out[l], d->layer_in[l]);
      for (i = 0; i < d->layer_out[l]; i++) dst[i] = logistic_func(dst[i]);
      src = dst;
      dst = (dst == bufa) ? bufb : bufa;
    }
    l = d->n_layers - 1;
    gemv(row, src, d->w[l], d->b[l], d->layer_out[l], d->layer_in[l]);
    logprob = oracle_addlog_array(row, d->out_dim);
    for (i = 0; i < d->out_dim; i++) row[i] = JB200_INV_LOG_TEN * (row[i] - logprob) - d->state_prior[i];
  }
  free(bufa); free(bufb);
  return 0;
}
