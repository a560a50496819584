/*
 * path_oracle.c -- CPU reference of KGEModel.path_rank_statistics / predict_path_topk, plain C.  TEST INFRASTRUCTURE.
 *
 * It compiles oracle/kge_oracle.c into the same unit, so the fold takes its phase scale and Cody-Waite sin/cos, and
 * ko_scores_from_q takes its score_row (the canonical blocked sum of DESIGN.md section 4) without restating them.
 * Build with -ffp-contract=off: every operation is a single correctly rounded IEEE operation.
 * tests/path_oracle.py builds and loads it; tests/test_path_cpu.py pins the fold to ko_query_vectors at L = 1 and to
 * float64 at L = 2..4.
 */
#include "../oracle/kge_oracle.c"

/* Path queries (DESIGN.md section 3.13): the fold of anchors [Q] along paths [Q, L] (hop r < nrelation forward, r +
 * nrelation inverted, -1 padding after the last hop) into qvec [Q, De].  Tail-batch: q = row(a) (pRotatE: row(a) / scale)
 * through hops 1..L; head-batch: q = row(a) (TransE -row(a), pRotatE -row(a) / scale) through hops L..1.  ComplEx and
 * RotatE multiply by r (build_q's tail formula with F = q) or by conj(r) (its head formula). */
void ko_path_query_vectors(int model, int head, const float *E, const float *R, int64_t nrelation, int De, int Dr,
                           float rho, const int64_t *anchors, const int64_t *paths, int64_t Q, int64_t L, float *qvec) {
  const int d = kdim(model, De);
  const float scale = phase_scale(model, rho);
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < Q; ++i) {
    const int64_t *row = paths + i * L;
    int64_t len = 0;
    while (len < L && row[len] != -1) ++len;
    const float *A = E + anchors[i] * De;
    float *q = qvec + i * De;
    for (int k = 0; k < d; ++k) {
      float q0 = A[k], q1 = (model == COMPLEX_ || model == ROTATE) ? A[d + k] : 0.f;
      if (model == PROTATE) q0 = q0 / scale;
      if (head && (model == TRANSE || model == PROTATE)) q0 = -q0;
      for (int64_t t = 0; t < len; ++t) {
        const int64_t h = row[head ? len - 1 - t : t];
        const int inv = h >= nrelation;
        const float *Rr = R + (inv ? h - nrelation : h) * Dr;
        switch (model) {
          case TRANSE:
            q0 = inv ? q0 - Rr[k] : (head ? Rr[k] + q0 : q0 + Rr[k]);
            break;
          case DISTMULT:
            q0 = head ? Rr[k] * q0 : q0 * Rr[k];
            break;
          case COMPLEX_: case ROTATE: {
            float rr, ri;
            if (model == COMPLEX_) { rr = Rr[k]; ri = Rr[d + k]; }
            else sincos_cw(Rr[k] / scale, &ri, &rr);
            float n0, n1;
            if (head == inv) { n0 = q0 * rr - q1 * ri; n1 = q0 * ri + q1 * rr; }
            else             { n0 = rr * q0 + ri * q1; n1 = rr * q1 - ri * q0; }
            q0 = n0; q1 = n1;
            break;
          }
          default: {
            const float pr = Rr[k] / scale;
            q0 = inv ? q0 - pr : (head ? pr + q0 : q0 + pr);
          }
        }
      }
      q[k] = q0;
      if (model == COMPLEX_ || model == ROTATE) q[d + k] = q1;
    }
  }
}

/* scores [Q, nentity] of every entity against the given query vectors qvec [Q, De] (score_row, no filter) */
void ko_scores_from_q(int model, int head, const float *E, int64_t nentity, int De, float gamma, float rho,
                      float modulus, const float *qvec, int64_t Q, float *scores) {
  const int d = kdim(model, De);
  const float scale = phase_scale(model, rho);
#pragma omp parallel for schedule(dynamic, 1)
  for (int64_t i = 0; i < Q; ++i)
    for (int64_t j = 0; j < nentity; ++j)
      scores[i * nentity + j] = score_row(model, head, qvec + i * De, E + j * De, d, gamma, scale, modulus);
}
