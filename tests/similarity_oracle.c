/*
 * similarity_oracle.c -- CPU reference of KGEModel.nearest_neighbors' scores, plain C.  TEST INFRASTRUCTURE.
 *
 * ko_similarity restates the canonical sequence of DESIGN.md section 3.12 so that the device scores can be compared
 * bit for bit: acc() cuts the k axis into blocks of 32, sums each block in index order from +0.0f and adds the block
 * sums in index order; every operation is a correctly rounded single IEEE operation (build with -ffp-contract=off).
 *   metric 0 dot     acc(q x)
 *   metric 1 cosine  acc(q x) / (|q| |x|),  |v| = sqrt(acc(v v))
 *   metric 2 l2      -sqrt(acc((q - x)^2))
 *   metric 3 l1      -acc(|q - x|)
 * tests/similarity_oracle.py builds and loads it; tests/test_similarity_oracle.py pins it to numpy and float64.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#define KB 32

static float term(int metric, float q, float x) {
  switch (metric) {
    case 2: { float t = q - x; return t * t; }
    case 3: return fabsf(q - x);
    default: return q * x;
  }
}

static float acc(int metric, const float *q, const float *x, int width) {
  float a = 0.f;
  for (int k0 = 0; k0 < width; k0 += KB) {
    float part = 0.f;
    const int k1 = k0 + KB < width ? k0 + KB : width;
    for (int k = k0; k < k1; ++k) part = part + term(metric, q[k], x[k]);
    a = a + part;
  }
  return a;
}

static float norm(const float *v, int width) { return sqrtf(acc(0, v, v, width)); }

/* out [Q, rows]: the score of every (query, row) pair */
void ko_similarity(const float *table, int64_t rows, int width, const float *queries, int64_t Q, int metric,
                   float *out) {
  float *xn = NULL;
  if (metric == 1) {
    xn = (float *)malloc(sizeof(float) * (size_t)(rows > 0 ? rows : 1));
#pragma omp parallel for schedule(static)
    for (int64_t j = 0; j < rows; ++j) xn[j] = norm(table + j * width, width);
  }
#pragma omp parallel for schedule(dynamic, 1)
  for (int64_t i = 0; i < Q; ++i) {
    const float *q = queries + i * width;
    const float qn = metric == 1 ? norm(q, width) : 0.f;
    for (int64_t j = 0; j < rows; ++j) {
      const float a = acc(metric, q, table + j * width, width);
      float s;
      switch (metric) {
        case 1: s = a / (qn * xn[j]); break;
        case 2: s = -sqrtf(a); break;
        case 3: s = -a; break;
        default: s = a;
      }
      out[i * rows + j] = s;
    }
  }
  free(xn);
}
