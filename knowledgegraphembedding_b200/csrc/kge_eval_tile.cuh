// kge_eval_tile.cuh -- the canonical score tile shared by the evaluation kernels (count_ranks_kernel in kge_eval.cu,
// topk_kernel in kge_eval_topk.cu; relation_tile_kernel in kge_eval_relation.cu reuses the element ops, the constants,
// the cp.async helpers and the top-k key): element ops, the canonical accumulation order, the cp.async staging of a
// [64 queries x 64 entities] tile and its k-loop.  Every kernel that runs tile_mainloop<OP, ALIGNED, false> computes the
// same score bits for a (query, entity) pair, which is what oracle/kge_oracle.c reproduces.
#pragma once
#include "kge_rows.cuh"

namespace kge {

// ---- exact element ops -----------------------------------------------------------------------------------
template <int OP>
__device__ __forceinline__ float op_exact(float q0, float q1, float x0, float x1) {
  if constexpr (OP == OP_SUBABS) return fabsf(fsub(q0, x0));                       // model.py:170,172
  else if constexpr (OP == OP_ADDABS) return fabsf(fadd(x0, q0));                  // model.py:168,172
  else if constexpr (OP == OP_MUL) return fmul(q0, x0);                            // model.py:177-179
  else if constexpr (OP == OP_CMUL) return fadd(fmul(q0, x0), fmul(q1, x1));       // model.py:192,196
  else if constexpr (OP == OP_CDIST) {                                             // model.py:217-226
    const float a = fsub(q0, x0), b = fsub(q1, x1);
    return fsqrt(ffma(b, b, fmul(a, a)));
  } else if constexpr (OP == OP_SUBSIN) return fabsf(sin_rep(fsub(q0, x0)));       // model.py:243-246 (x = phase table)
  else if constexpr (OP == OP_ADDSIN) return fabsf(sin_rep(fadd(x0, q0)));         // model.py:241
  else {                                                                           // similarity search, l2
    const float t = fsub(q0, x0);
    return fmul(t, t);
  }
}

// Fast (non-canonical) element op of the two-stage RotatE evaluation: contraction allowed, one-instruction
// approximate sqrt.  Per-term relative deviation from op_exact is below 2^-20 (sqrt.approx <= 2^-21, the a^2+b^2
// association <= 2^-22, exact rounding <= 2^-24); see kFastBand.
// pRotatE: |sin(t)| has period pi, so t is reduced by the nearest multiple of pi (two-constant Cody-Waite: the product
// k * 3.140625 is exact for |k| < 2^15; each of the two FMAs rounds once, <= 1.2e-7 for |r| <= 2; the residual constant
// is good to 2^-24 relative, i.e. <= |k| * 6e-11) to r in [-pi/2, pi/2], where sin.approx (one MUFU instruction) is
// within 2^-20.9 = 5.1e-7 of sin (PTX ISA, quadrant 00): 8 instructions instead of the ~35 of sin_rep.  For |t| < 4e4
// (|k| < 1.3e4) the reduction error is <= 2.4e-7 + 8e-7; beyond that the result is NaN, which the epilogue turns into
// "undecidable" (exact re-score), never into a wrong count.
__device__ __forceinline__ float abs_sin_fast(float t) {
  const float k = rintf(t * 0.318309886183790672f);
  float r = fmaf(-k, 3.140625f, t);
  r = fmaf(-k, 9.67653589793e-4f, r);
  float s;
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(r));
  return fabsf(t) < 4.0e4f ? fabsf(s) : __int_as_float(0x7fc00000);
}
template <int OP>
__device__ __forceinline__ float op_fast(float q0, float q1, float x0, float x1) {
  static_assert(OP == OP_CDIST || OP == OP_SUBSIN || OP == OP_ADDSIN, "ops with a fast variant");
  if constexpr (OP == OP_CDIST) {
    const float a = q0 - x0, b = q1 - x1;
    return sqrt_approx(fmaf(a, a, b * b));
  } else if constexpr (OP == OP_SUBSIN) return abs_sin_fast(q0 - x0);
  else return abs_sin_fast(x0 + q0);
}
// Band of the two-stage pass: |s_fast - s_canonical| <= eps(s_fast) = c_abs + c_rel * |gamma - s_fast| + c_ulp * |s_fast|
// (fast_band / fast_eps below; kge_eval_two_stage_band exports the coefficients).  Both scores are
// s = fl(gamma - p), p = acc (RotatE) or fl(acc * modulus) (pRotatE), of two different sums acc_f and acc_c.
//  * c_rel, the sums.  RotatE: 2^-20 per term + two blocked fp32 sums of the same blocks (each within (32 + d/32) * 2^-24
//    <= 6e-6 of the exact sum for d <= 2048), rounded up: kFastBand.  pRotatE: the same two sums (1.15e-5) and the two
//    roundings of acc * modulus (1.2e-7) fit in kFastSinSum; its per-term error is absolute, c_abs = |modulus| d kFastSinTerm.
//  * c_ulp, the final subtraction.  fl(x) = x (1 + e) with |e| <= 2^-24 gives |s - (gamma - p)| <= 2^-24 |s| for s_f and
//    for s_c, and |s_c| <= |s_f| + eps, so the two roundings add 2^-23 |s_f| (+ 2^-24 eps, second order).  This term does
//    not shrink with |p_f - p_c|: sums that straddle a rounding boundary of gamma - p give scores one ulp of s apart however
//    close they are, while c_rel * |gamma - s| falls below that ulp once acc < ulp(gamma) / c_rel (0.12 at gamma = 24).
//    kFastUlp = 2^-22 takes it twice: the margin covers |gamma - s_f| underestimating |p_f| by up to 2^-24 |s_f| (times
//    c_rel) and the fp32 evaluation of eps (a few ulps of eps).
constexpr float kFastBand = 1.6e-5f;
// pRotatE: per term |fast - canonical| <= 5.1e-7 + 1.04e-6 (above) + 1.8e-7 (sin_rep's own 1.5 ulp) < kFastSinTerm; sums as above
constexpr float kFastSinTerm = 2.0e-6f, kFastSinSum = 1.2e-5f;
constexpr float kFastUlp = 0x1p-22f;
constexpr int kFastMaxD = 2048;                            // the sum bounds above hold up to this d
struct FastBand {
  float c_abs, c_rel, c_ulp;
};
KGE_HD FastBand fast_band(bool protate, int d, float modulus) {
  if (protate) return FastBand{fabsf(modulus) * (float)d * kFastSinTerm + 1e-12f, kFastSinSum, kFastUlp};
  return FastBand{1e-12f, kFastBand, kFastUlp};
}
KGE_HD float fast_eps(const FastBand &b, float gamma, float s) {
  return b.c_abs + b.c_rel * fabsf(gamma - s) + b.c_ulp * fabsf(s);
}

template <int OP>
__device__ __forceinline__ float finish_exact(float acc, float gamma, float modulus) {
  if constexpr (OP == OP_MUL || OP == OP_CMUL) return acc;
  else if constexpr (OP == OP_SUBSIN || OP == OP_ADDSIN) return fsub(gamma, fmul(acc, modulus));
  else return fsub(gamma, acc);
}

// Accumulation order of every evaluation score (the "canonical order", DESIGN.md section 4): the k axis is cut
// into blocks of KC consecutive indices; each block is summed in index order from 0.0f, and the block sums are
// added in index order.  (Error grows with sqrt(KC) + sqrt(d/KC) instead of sqrt(d).)
constexpr int TQ = 64, TJ = 64, KC = 32, ST = KC + 4, EVAL_THREADS = 256;

// ---- tile staging ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(float *smem_dst, const float *gsrc, bool valid) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int bytes = valid ? 16 : 0;                       // src-size 0 => 16 bytes of zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct EvalArgs {
  const float *qvec;            // [Q, De]
  const float *X;               // candidate table [nentity, De] (entity table, or phase table for pRotatE)
  const int64_t *queries;       // [Q, 3]
  const float *pos_score;       // [Q]
  const uint32_t *filter_bits;  // [Q, words]
  int32_t *counts;              // [Q]
  float *scores_out;            // [Q, nentity] or null: the score each pair was decided on (the fast one in a FAST pass)
  const float *modulus;
  int64_t Q, nentity, ent_begin, ent_end;
  int d, De, pos_col, words;
  float gamma;
  int2 *amb;                    // two-stage mode: ambiguous (q, j) pairs for the exact re-score
  int *amb_count;               // [0] appended, [1] overflow
  int amb_capacity;
};

// Stage one k-chunk of the query tile and the entity tile:  smem[row][half][ST]
template <bool CPLX, bool ALIGNED>
__device__ __forceinline__ void stage_tiles(const EvalArgs &a, float *sq, float *sx, int64_t q0, int64_t j0, int k0) {
  constexpr int H = CPLX ? 2 : 1;
  constexpr int VPR = KC / 4;                              // float4 per row-half per chunk
  constexpr int TOTAL = (TQ + TJ) * H * VPR;
  for (int idx = threadIdx.x; idx < TOTAL; idx += EVAL_THREADS) {
    const int v = idx % VPR;
    const int h = (idx / VPR) % H;
    const int row = idx / (VPR * H);
    const int k = k0 + v * 4;
    const bool is_q = row < TQ;
    int64_t g = is_q ? q0 + row : j0 + (row - TQ);
    const int64_t lim = is_q ? a.Q : a.ent_end;
    if (g >= lim) g = lim - 1;                             // clamp: the duplicate row's results are masked out
    const float *src = (is_q ? a.qvec : a.X) + g * a.De + h * a.d + k;
    float *dst = (is_q ? sq + row * (H * ST) : sx + (row - TQ) * (H * ST)) + h * ST + v * 4;
    if constexpr (ALIGNED) {
      cp_async16(dst, k < a.d ? src : (is_q ? a.qvec : a.X), k < a.d);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) dst[e] = (k + e < a.d) ? src[e] : 0.f;
    }
  }
}

// ---- k-loop of one [TQ x TJ] tile -------------------------------------------------------------------------------
// Returns v[i][j] = score accumulator (before finish_exact) of query q0 + tq + 16 i against entity j0 + tj + 16 j.
// smem holds two stages of [TQ + TJ][H][ST] floats.  The loop ends with __syncthreads(), so the caller may reuse smem.
// (The accumulators come back by value: through a reference parameter the function is simplified on its own before
// it is inlined, and the loop is scheduled differently inside the kernels.)
struct TileAcc {
  float v[4][4];
};
template <int OP, bool ALIGNED, bool FAST = false>
__device__ __forceinline__ TileAcc tile_mainloop(const EvalArgs &a, float *smem, int64_t q0, int64_t j0, int tq, int tj) {
  float acc[4][4];
  constexpr bool CPLX = op_is_complex(OP);
  constexpr int H = CPLX ? 2 : 1;
  constexpr int TILE_Q = TQ * H * ST, TILE_X = TJ * H * ST;
  constexpr int STAGE = TILE_Q + TILE_X;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int nchunks = (a.d + KC - 1) / KC;
  stage_tiles<CPLX, ALIGNED>(a, smem, smem + TILE_Q, q0, j0, 0);
  cp_async_commit();
  for (int c = 0; c < nchunks; ++c) {
    const int cur = c & 1;
    if (c + 1 < nchunks)
      stage_tiles<CPLX, ALIGNED>(a, smem + (cur ^ 1) * STAGE, smem + (cur ^ 1) * STAGE + TILE_Q, q0, j0, (c + 1) * KC);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const float *Q_ = smem + cur * STAGE, *X_ = Q_ + TILE_Q;
    float part[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) part[i][j] = 0.f;
    constexpr bool PACKED = FAST && OP == OP_CDIST;        // FADD2 / FMUL2 / FFMA2: 3.5 issue slots per term, not 6
    f2 part2[PACKED ? 4 : 1][PACKED ? 4 : 1];
    if constexpr (PACKED) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) part2[i][j] = pack2(0.f, 0.f);
    }
#pragma unroll 2
    for (int kk = 0; kk < KC; kk += 4) {
      float4 qa[4], qb[4], xa[4], xb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        qa[i] = *reinterpret_cast<const float4 *>(Q_ + (tq + 16 * i) * (H * ST) + kk);
        xa[i] = *reinterpret_cast<const float4 *>(X_ + (tj + 16 * i) * (H * ST) + kk);
        if constexpr (CPLX) {
          qb[i] = *reinterpret_cast<const float4 *>(Q_ + (tq + 16 * i) * (H * ST) + ST + kk);
          xb[i] = *reinterpret_cast<const float4 *>(X_ + (tj + 16 * i) * (H * ST) + ST + kk);
        } else {
          qb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          xb[i] = qb[i];
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {       // k ascending inside the group => index-order accumulation
          if constexpr (PACKED) {
            // |q - x| for four k at once: differences, squares and the partial sums run on packed pairs; only the four
            // square roots (MUFU) are scalar.  The approximate scores stay inside the band of the two-stage scheme
            // (same per-term error; the block sum is formed as (even k) + (odd k), still at most KC terms deep).
            const f2 a01 = sub2(pack2(qa[i].x, qa[i].y), pack2(xa[j].x, xa[j].y));
            const f2 a23 = sub2(pack2(qa[i].z, qa[i].w), pack2(xa[j].z, xa[j].w));
            const f2 b01 = sub2(pack2(qb[i].x, qb[i].y), pack2(xb[j].x, xb[j].y));
            const f2 b23 = sub2(pack2(qb[i].z, qb[i].w), pack2(xb[j].z, xb[j].w));
            const f2 m01 = fma2(b01, b01, mul2(a01, a01));
            const f2 m23 = fma2(b23, b23, mul2(a23, a23));
            float s0, s1, s2, s3;
            unpack2(m01, s0, s1);
            unpack2(m23, s2, s3);
            const f2 r01 = pack2(sqrt_approx(s0), sqrt_approx(s1));
            const f2 r23 = pack2(sqrt_approx(s2), sqrt_approx(s3));
            part2[i][j] = add2(part2[i][j], add2(r01, r23));
          } else if constexpr (FAST) {
            part[i][j] += op_fast<OP>(qa[i].x, qb[i].x, xa[j].x, xb[j].x);
            part[i][j] += op_fast<OP>(qa[i].y, qb[i].y, xa[j].y, xb[j].y);
            part[i][j] += op_fast<OP>(qa[i].z, qb[i].z, xa[j].z, xb[j].z);
            part[i][j] += op_fast<OP>(qa[i].w, qb[i].w, xa[j].w, xb[j].w);
          } else {
            part[i][j] = fadd(part[i][j], op_exact<OP>(qa[i].x, qb[i].x, xa[j].x, xb[j].x));
            part[i][j] = fadd(part[i][j], op_exact<OP>(qa[i].y, qb[i].y, xa[j].y, xb[j].y));
            part[i][j] = fadd(part[i][j], op_exact<OP>(qa[i].z, qb[i].z, xa[j].z, xb[j].z));
            part[i][j] = fadd(part[i][j], op_exact<OP>(qa[i].w, qb[i].w, xa[j].w, xb[j].w));
          }
        }
    }
    if constexpr (PACKED) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float lo, hi;
          unpack2(part2[i][j], lo, hi);
          part[i][j] = lo + hi;
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fadd(acc[i][j], part[i][j]);
    __syncthreads();
  }
  TileAcc r;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) r.v[i][j] = acc[i][j];
  return r;
}

// Top-k candidate key (kge_eval_topk.cu, kge_eval_relation.cu): (orderable(score) << 32) | (0xFFFFFFFF - id), so that a
// larger key is a better candidate -- score descending, then id ascending, NaN last, -0.0 == +0.0.  Key 0 is an empty slot.
__device__ __forceinline__ uint64_t topk_key(float s, int64_t id) {
  uint32_t ord = 0;                                        // NaN: below every number
  if (!(s != s)) {
    const uint32_t u = __float_as_uint(s == 0.f ? 0.f : s);  // -0.0 -> +0.0
    ord = (u & 0x80000000u) ? ~u : (u | 0x80000000u);     // -inf -> 0x007FFFFF > 0
  }
  return ((uint64_t)ord << 32) | (uint64_t)(0xFFFFFFFFu - (uint32_t)id);
}

static inline int eval_mode(int mode, bool &head) {
  if (mode == KGE_HEAD_BATCH) head = true;
  else if (mode == KGE_TAIL_BATCH) head = false;
  else {
    set_error("negative batch mode %d not supported", mode);     // dataloader.py:147
    return KGE_ERR_INVALID;
  }
  return KGE_OK;
}

static inline int fill_eval_args(const kge_model_t *m, bool head, const float *qvec, const int64_t *queries, int64_t Q,
                                 const float *phase_table, EvalArgs &a) {
  const bool cplx = m->model == KGE_COMPLEX || m->model == KGE_ROTATE;
  KGE_REQUIRE(m->model != KGE_PROTATE || phase_table, "pRotatE evaluation needs kge_eval_phase_table");
  a.qvec = qvec;
  a.X = m->model == KGE_PROTATE ? phase_table : m->entity;
  a.queries = queries;
  a.modulus = m->modulus;
  a.Q = Q;
  a.nentity = m->nentity;
  a.d = cplx ? (int)(m->entity_dim / 2) : (int)m->entity_dim;
  a.De = (int)m->entity_dim;
  a.pos_col = head ? 0 : 2;
  a.words = (int)((m->nentity + 31) / 32);
  a.gamma = m->gamma;
  return KGE_OK;
}

// 16-byte cp.async staging needs aligned rows and operands
static inline bool eval_aligned(const EvalArgs &a) {
  return (a.d % 4 == 0) && (a.De % 4 == 0) && ((((uintptr_t)a.qvec | (uintptr_t)a.X) & 15) == 0);
}

}  // namespace kge
