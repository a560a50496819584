// kge_eval_relation.cu -- relation prediction: which relation links h to t.  Every query (h, ?, t) is scored against
// every relation r with the 'single'-mode score of (h, r, t) in the canonical order, i.e. the bits of column t of the
// tail-batch entity scores of (h, r, ?) (count_ranks_kernel, topk_kernel) and of oracle/kge_oracle.c's ko_forward.
//
//   relation_table_kernel  the relation operand of every relation, once per call: (cos | sin) of R / scale for
//                          RotatE (build_q's sincos_rep), R / scale for pRotatE; the other models use R as it is.
//   relation_tile_kernel   grid (relation tiles of 64 x query tiles of 64).  The entity kernels fold q = fold(h, r) once
//                          per query and stream candidate rows against it; here the candidate is the relation, so the
//                          fold runs per (query, relation, k) term: per k-chunk the h rows, the t rows and the relation
//                          operand rows are staged with the cp.async double buffer of kge_eval_tile.cuh, then every term
//                          is build_q's tail-batch fold followed by op_exact, summed in the canonical blocks of KC.
//                          Epilogue COUNT: count_ranks_kernel's comparison with the positive (relation queries[q*3+1]),
//                          filter bitmap [Q, ceil(nrelation/32)], integer counts.  Epilogue KEYS: topk_key of every
//                          relation of the slice into a [Q, L*k] key matrix (key 0: excluded or padding), which
//                          topk_merge_kernel (kge_eval_topk_merge) reduces to the k best with L lists per query.
//   relation_lookup_kernel the relation filter bitmap from the sorted-key index h*nentity + t -> relations.
#include "kge_eval_tile.cuh"

namespace kge {

// ---- relation operand table ---------------------------------------------------------------------------------------
template <int MODEL>
__global__ void relation_table_kernel(const float *__restrict__ R, int64_t nrelation, int d, int Dr, float scale,
                                      float *__restrict__ out) {
  const int64_t n = nrelation * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / d;
    const int k = (int)(i - r * d);
    if constexpr (MODEL == KGE_ROTATE) {                   // build_q: sincos_rep(fdiv(Rr[k], scale), &s, &c)
      float s, c;
      sincos_rep(fdiv(R[r * Dr + k], scale), &s, &c);
      out[r * 2 * d + k] = c;
      out[r * 2 * d + d + k] = s;
    } else {                                               // pRotatE: build_q's pr = fdiv(Rr[k], scale)
      out[r * d + k] = fdiv(R[r * Dr + k], scale);
    }
  }
}

// ---- tail-batch fold of build_q (kge_rows.cuh) on register operands: f = head row, (r0, r1) = relation operand ------
template <int MODEL>
__device__ __forceinline__ void fold_tail(float f0, float f1, float r0, float r1, float &q0, float &q1) {
  if constexpr (MODEL == KGE_TRANSE) q0 = fadd(f0, r0);                                  // h + r
  else if constexpr (MODEL == KGE_DISTMULT) q0 = fmul(f0, r0);                           // h * r
  else if constexpr (MODEL == KGE_COMPLEX) {
    q0 = fsub(fmul(f0, r0), fmul(f1, r1));
    q1 = fadd(fmul(f0, r1), fmul(f1, r0));
  } else if constexpr (MODEL == KGE_ROTATE) {                                            // (r0, r1) = (cos, sin)
    q0 = fsub(fmul(f0, r0), fmul(f1, r1));
    q1 = fadd(fmul(f0, r1), fmul(f1, r0));
  } else q0 = fadd(f0, r0);                                                              // pRotatE: ph + pr
}

struct RelArgs {
  const float *E;               // entity side [nentity, De]: entity table, or phase table for pRotatE
  const float *Rop;             // relation operand [nrelation, Dro]
  const int64_t *queries;       // [Q, 3]
  const float *pos_score;       // COUNT: [Q]
  const uint32_t *bits;         // COUNT: filter, KEYS: exclusion (may be null); [Q, words]
  int32_t *counts;              // COUNT: [Q]
  float *scores_out;            // COUNT: [Q, nrelation] or null
  uint64_t *keys;               // KEYS: [Q, key_row]
  int32_t *err;                 // KEYS: bad-id flag (may be null)
  const float *modulus;
  int64_t Q, nentity, nrelation, rel_begin, rel_end, key_row;
  int d, De, Dro, words;
  float gamma;
};

constexpr int EPI_COUNT = 0, EPI_KEYS = 1;

template <int MODEL>
__host__ __device__ constexpr int relation_halves() { return MODEL == KGE_COMPLEX || MODEL == KGE_ROTATE ? 2 : 1; }

// One k-chunk: smem[row][half][ST] for the h rows, the t rows (HE halves) and the relation rows (HR halves).
template <int HE, int HR, bool ALIGNED>
__device__ __forceinline__ void stage_relation(const RelArgs &a, const int64_t *ids, float *sh, float *sr, int64_t r0,
                                               int k0) {
  constexpr int VPR = KC / 4;
  constexpr int QSIDE = 2 * TQ * HE;                       // h rows then t rows
  constexpr int TOTAL = (QSIDE + TJ * HR) * VPR;
  for (int idx = threadIdx.x; idx < TOTAL; idx += EVAL_THREADS) {
    const int v = idx % VPR;
    const int rest = idx / VPR;
    const int k = k0 + v * 4;
    const float *base;
    const float *src;
    float *dst;
    if (rest < QSIDE) {
      const int row = rest / HE, h = rest % HE;            // row < TQ: head of query row, else tail of query row - TQ
      base = a.E;
      src = a.E + ids[row] * a.De + h * a.d + k;
      dst = sh + row * (HE * ST) + h * ST + v * 4;
    } else {
      const int row = (rest - QSIDE) / HR, h = (rest - QSIDE) % HR;
      int64_t g = r0 + row;
      if (g >= a.rel_end) g = a.rel_end - 1;               // clamp: the duplicate row's results are masked out
      base = a.Rop;
      src = a.Rop + g * a.Dro + h * a.d + k;
      dst = sr + row * (HR * ST) + h * ST + v * 4;
    }
    if constexpr (ALIGNED) {
      cp_async16(dst, k < a.d ? src : base, k < a.d);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) dst[e] = (k + e < a.d) ? src[e] : 0.f;
    }
  }
}

// Occupancy: 2 CTAs per SM for every model.  The complex models stage 2 x 2 query-side halves and 2 relation halves per
// chunk, 110.6 KB of shared memory per CTA for both stages, so two CTAs fit the 228 KB of an SM; the other models need
// half of that.  Registers are capped at 128 per thread by the launch bounds; ptxas reports no spills for any
// instantiation (DESIGN.md section 3.9).
template <int MODEL, bool ALIGNED, int EPI>
__global__ void __launch_bounds__(EVAL_THREADS, 2) relation_tile_kernel(const RelArgs a) {
  constexpr int OP = op_of(MODEL, false);
  constexpr int HE = op_is_complex(OP) ? 2 : 1;
  constexpr int HR = relation_halves<MODEL>();
  constexpr int TILE_Q = 2 * TQ * HE * ST, TILE_R = TJ * HR * ST;
  constexpr int STAGE = TILE_Q + TILE_R;
  extern __shared__ __align__(16) float smem[];
  __shared__ int64_t ids[2 * TQ];                          // head ids, then tail ids of the tile's queries
  __shared__ int cnt_sh[TQ];

  const int tid = threadIdx.x;
  const int tq = tid % 16, tj = tid / 16;
  const int64_t r0 = a.rel_begin + (int64_t)blockIdx.x * TJ;
  const int64_t q0 = (int64_t)blockIdx.y * TQ;
  if (tid < 2 * TQ) {
    const int64_t qi = q0 + (tid % TQ);
    int64_t e = 0;
    if (qi < a.Q) {
      e = a.queries[qi * 3 + (tid < TQ ? 0 : 2)];
      if ((uint64_t)e >= (uint64_t)a.nentity) {
        if (a.err) *a.err = 1;
        e = 0;
      }
    }
    ids[tid] = e;
  }
  if (tid < TQ) cnt_sh[tid] = 0;
  __syncthreads();

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int nchunks = (a.d + KC - 1) / KC;
  stage_relation<HE, HR, ALIGNED>(a, ids, smem, smem + TILE_Q, r0, 0);
  cp_async_commit();
  for (int c = 0; c < nchunks; ++c) {
    const int cur = c & 1;
    if (c + 1 < nchunks)
      stage_relation<HE, HR, ALIGNED>(a, ids, smem + (cur ^ 1) * STAGE, smem + (cur ^ 1) * STAGE + TILE_Q, r0,
                                      (c + 1) * KC);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const float *H_ = smem + cur * STAGE, *T_ = H_ + TQ * HE * ST, *R_ = H_ + TILE_Q;
    float part[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) part[i][j] = 0.f;
#pragma unroll 1
    for (int kk = 0; kk < KC; kk += 4) {
      float4 ra[4], rb[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        ra[j] = *reinterpret_cast<const float4 *>(R_ + (tj + 16 * j) * (HR * ST) + kk);
        rb[j] = HR == 2 ? *reinterpret_cast<const float4 *>(R_ + (tj + 16 * j) * (HR * ST) + ST + kk)
                        : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float *hrow = H_ + (tq + 16 * i) * (HE * ST) + kk, *trow = T_ + (tq + 16 * i) * (HE * ST) + kk;
        const float4 ha = *reinterpret_cast<const float4 *>(hrow), ta = *reinterpret_cast<const float4 *>(trow);
        float4 hb = make_float4(0.f, 0.f, 0.f, 0.f), tb = hb;
        if constexpr (HE == 2) {
          hb = *reinterpret_cast<const float4 *>(hrow + ST);
          tb = *reinterpret_cast<const float4 *>(trow + ST);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {       // k ascending inside the group => index-order accumulation
          float q0v = 0.f, q1v = 0.f;
          fold_tail<MODEL>(ha.x, hb.x, ra[j].x, rb[j].x, q0v, q1v);
          part[i][j] = fadd(part[i][j], op_exact<OP>(q0v, q1v, ta.x, tb.x));
          fold_tail<MODEL>(ha.y, hb.y, ra[j].y, rb[j].y, q0v, q1v);
          part[i][j] = fadd(part[i][j], op_exact<OP>(q0v, q1v, ta.y, tb.y));
          fold_tail<MODEL>(ha.z, hb.z, ra[j].z, rb[j].z, q0v, q1v);
          part[i][j] = fadd(part[i][j], op_exact<OP>(q0v, q1v, ta.z, tb.z));
          fold_tail<MODEL>(ha.w, hb.w, ra[j].w, rb[j].w, q0v, q1v);
          part[i][j] = fadd(part[i][j], op_exact<OP>(q0v, q1v, ta.w, tb.w));
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fadd(acc[i][j], part[i][j]);
    __syncthreads();
  }

  // ---- epilogue ---------------------------------------------------------------------------------------------------
  const float modulus = a.modulus ? a.modulus[0] : 1.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t qi = q0 + tq + 16 * i;
    if (qi >= a.Q) continue;
    if constexpr (EPI == EPI_COUNT) {                      // count_ranks_kernel's epilogue, relations as candidates
      const float sp = a.pos_score[qi];
      const int64_t pid = a.queries[qi * 3 + 1];
      int c = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t rj = r0 + tj + 16 * j;
        if (rj >= a.rel_end) continue;
        float s = finish_exact<OP>(acc[i][j], a.gamma, modulus);
        const bool filtered = rj != pid && ((a.bits[qi * a.words + (rj >> 5)] >> (rj & 31)) & 1u);
        if (filtered) s = fadd(sp, -1.0f);                 // candidate replaced by the positive, bias -1
        else if (rj != pid) c += (s > sp) || (s == sp && rj < pid);
        if (a.scores_out) a.scores_out[qi * a.nrelation + rj] = s;
      }
      if (c) atomicAdd(&cnt_sh[tq + 16 * i], c);
    } else {                                               // key of every relation; excluded ones keep the zeroed slot
      const uint32_t *ex = a.bits ? a.bits + qi * a.words : nullptr;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t rj = r0 + tj + 16 * j;
        if (rj >= a.rel_end) continue;
        if (ex && ((ex[rj >> 5] >> (rj & 31)) & 1u)) continue;
        a.keys[qi * a.key_row + (rj - a.rel_begin)] = topk_key(finish_exact<OP>(acc[i][j], a.gamma, modulus), rj);
      }
    }
  }
  if constexpr (EPI == EPI_COUNT) {
    __syncthreads();
    if (tid < TQ && cnt_sh[tid] && q0 + tid < a.Q) atomicAdd(&a.counts[q0 + tid], cnt_sh[tid]);
  }
}

// Relation filter bitmap from the sorted-key index (keys h*nentity + t, runs of relation ids): one thread per query.
__global__ void relation_lookup_kernel(const int64_t *__restrict__ keys, const int64_t *__restrict__ key_offsets,
                                       const int32_t *__restrict__ relations, int64_t nkeys,
                                       const int64_t *__restrict__ queries, int64_t Q, int64_t nentity,
                                       int64_t nrelation, int words, uint32_t *__restrict__ bits) {
  for (int64_t qi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; qi < Q; qi += (int64_t)gridDim.x * blockDim.x) {
    const int64_t h = queries[qi * 3], t = queries[qi * 3 + 2];
    if ((uint64_t)h >= (uint64_t)nentity || (uint64_t)t >= (uint64_t)nentity) continue;   // flagged by the score kernels
    const int64_t key = h * nentity + t;
    int64_t lo = 0, hi = nkeys;                            // lower bound
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (lo == nkeys || keys[lo] != key) continue;
    for (int64_t i = key_offsets[lo]; i < key_offsets[lo + 1]; ++i) {
      const int32_t r = relations[i];
      if (r >= 0 && r < nrelation) atomicOr(&bits[qi * words + (r >> 5)], 1u << (r & 31));
    }
  }
}

template <int MODEL, int EPI>
static int launch_relation(const RelArgs &a, bool aligned, cudaStream_t st) {
  constexpr int HE = op_is_complex(op_of(MODEL, false)) ? 2 : 1;
  const size_t smem = sizeof(float) * 2 * (2 * TQ * HE + TJ * relation_halves<MODEL>()) * ST;
  const dim3 grid((unsigned)((a.rel_end - a.rel_begin + TJ - 1) / TJ), (unsigned)((a.Q + TQ - 1) / TQ));
  auto kern = aligned ? relation_tile_kernel<MODEL, true, EPI> : relation_tile_kernel<MODEL, false, EPI>;
  KGE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, EVAL_THREADS, smem, st>>>(a);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

template <int EPI>
static int dispatch_relation(int model, const RelArgs &a, cudaStream_t st) {
  const bool aligned = (a.d % 4 == 0) && (a.De % 4 == 0) && (a.Dro % 4 == 0) &&
                       ((((uintptr_t)a.E | (uintptr_t)a.Rop) & 15) == 0);
  switch (model) {
    case KGE_TRANSE: return launch_relation<KGE_TRANSE, EPI>(a, aligned, st);
    case KGE_DISTMULT: return launch_relation<KGE_DISTMULT, EPI>(a, aligned, st);
    case KGE_COMPLEX: return launch_relation<KGE_COMPLEX, EPI>(a, aligned, st);
    case KGE_ROTATE: return launch_relation<KGE_ROTATE, EPI>(a, aligned, st);
    default: return launch_relation<KGE_PROTATE, EPI>(a, aligned, st);
  }
}

static int relation_check(const kge_model_t *m, int64_t Q, int64_t rel_begin, int64_t rel_end) {
  const int rc = check_model(m);
  if (rc) return rc;
  KGE_REQUIRE(Q >= 0 && (Q + TQ - 1) / TQ <= 65535, "at most %d queries per call", 65535 * TQ);
  KGE_REQUIRE(rel_begin >= 0 && rel_begin <= rel_end && rel_end <= m->nrelation,
              "relation slice [%lld,%lld) outside [0,%lld)", (long long)rel_begin, (long long)rel_end,
              (long long)m->nrelation);
  return KGE_OK;
}

// The model's operands of the relation kernel; rel_table is required for RotatE and pRotatE, phase_table for pRotatE.
static int fill_relation_args(const kge_model_t *m, const int64_t *queries, int64_t Q, const float *rel_table,
                              const float *phase_table, int64_t rel_begin, int64_t rel_end, RelArgs &a) {
  const bool cplx = m->model == KGE_COMPLEX || m->model == KGE_ROTATE;
  const bool table = m->model == KGE_ROTATE || m->model == KGE_PROTATE;
  KGE_REQUIRE(queries, "null pointer");
  KGE_REQUIRE(!table || rel_table, "RotatE / pRotatE relation prediction needs kge_eval_relation_table");
  KGE_REQUIRE(m->model != KGE_PROTATE || phase_table, "pRotatE evaluation needs kge_eval_phase_table");
  a.E = m->model == KGE_PROTATE ? phase_table : m->entity;
  a.Rop = table ? rel_table : m->relation;
  a.queries = queries;
  a.modulus = m->modulus;
  a.Q = Q;
  a.nentity = m->nentity;
  a.nrelation = m->nrelation;
  a.rel_begin = rel_begin;
  a.rel_end = rel_end;
  a.d = cplx ? (int)(m->entity_dim / 2) : (int)m->entity_dim;
  a.De = (int)m->entity_dim;
  a.Dro = m->model == KGE_ROTATE ? 2 * a.d : m->model == KGE_PROTATE ? a.d : (int)m->relation_dim;
  a.words = (int)((m->nrelation + 31) / 32);
  a.gamma = m->gamma;
  return KGE_OK;
}

static size_t relation_keys_bytes(int64_t Q, int64_t rel_begin, int64_t rel_end, int k) {
  if (Q == 0 || rel_begin == rel_end) return 0;
  const int64_t lists = (rel_end - rel_begin + k - 1) / k;
  return sizeof(uint64_t) * (size_t)Q * (size_t)(lists * k);
}

}  // namespace kge

using namespace kge;

extern "C" int kge_eval_relation_table(const kge_model_t *m, float *rel_table, void *stream) {
  int rc = check_model(m);
  if (rc) return rc;
  if (m->model != KGE_ROTATE && m->model != KGE_PROTATE) return KGE_OK;       // R is used as it is
  KGE_REQUIRE(rel_table, "null pointer");
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  const int d = m->model == KGE_ROTATE ? (int)(m->entity_dim / 2) : (int)m->entity_dim;
  const int64_t n = m->nrelation * d;
  const int grid = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (m->model == KGE_ROTATE)
    relation_table_kernel<KGE_ROTATE><<<grid, 256, 0, st>>>(m->relation, m->nrelation, d, (int)m->relation_dim,
                                                           phase_scale(m), rel_table);
  else
    relation_table_kernel<KGE_PROTATE><<<grid, 256, 0, st>>>(m->relation, m->nrelation, d, (int)m->relation_dim,
                                                            phase_scale(m), rel_table);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

extern "C" int kge_eval_relation_count_ranks(const kge_model_t *m, const int64_t *queries, int64_t Q,
                                             const float *rel_table, const float *phase_table, const float *pos_score,
                                             const uint32_t *filter_bits, int64_t rel_begin, int64_t rel_end,
                                             int32_t *counts, float *scores_out, void *stream) {
  int rc = relation_check(m, Q, rel_begin, rel_end);
  if (rc) return rc;
  KGE_REQUIRE(queries && pos_score && filter_bits && counts, "null pointer");
  RelArgs a{};
  if ((rc = fill_relation_args(m, queries, Q, rel_table, phase_table, rel_begin, rel_end, a))) return rc;
  if (Q == 0 || rel_begin == rel_end) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  a.pos_score = pos_score;
  a.bits = filter_bits;
  a.counts = counts;
  a.scores_out = scores_out;
  return dispatch_relation<EPI_COUNT>(m->model, a, (cudaStream_t)stream);
}

extern "C" int64_t kge_eval_relation_topk_scratch_bytes(const kge_model_t *m, int64_t Q, int64_t rel_begin,
                                                        int64_t rel_end, int k) {
  const int rc = relation_check(m, Q, rel_begin, rel_end);
  if (rc) return rc;
  KGE_REQUIRE(k >= 1 && k <= KGE_TOPK_MAX, "k = %d outside [1, %d]", k, KGE_TOPK_MAX);
  return (int64_t)relation_keys_bytes(Q, rel_begin, rel_end, k);
}

extern "C" int kge_eval_relation_topk(const kge_model_t *m, const int64_t *queries, int64_t Q, const float *rel_table,
                                      const float *phase_table, const uint32_t *exclude_bits, int64_t rel_begin,
                                      int64_t rel_end, int k, uint64_t *keys_out, void *scratch, int64_t scratch_bytes,
                                      int32_t *err_flag, void *stream) {
  int rc = relation_check(m, Q, rel_begin, rel_end);
  if (rc) return rc;
  KGE_REQUIRE(k >= 1 && k <= KGE_TOPK_MAX, "k = %d outside [1, %d]", k, KGE_TOPK_MAX);
  KGE_REQUIRE(keys_out, "null pointer");
  RelArgs a{};
  if ((rc = fill_relation_args(m, queries, Q, rel_table, phase_table, rel_begin, rel_end, a))) return rc;
  const size_t need = relation_keys_bytes(Q, rel_begin, rel_end, k);
  KGE_REQUIRE(scratch_bytes >= (int64_t)need && (scratch || need == 0), "scratch of %lld bytes, need %lld",
              (long long)scratch_bytes, (long long)need);
  if (Q == 0) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (rel_begin == rel_end) {                              // nothing to select from: every slot empty
    KGE_CUDA_OK(cudaMemsetAsync(keys_out, 0, sizeof(uint64_t) * (size_t)Q * k, st));
    return KGE_OK;
  }
  a.bits = exclude_bits;
  a.keys = (uint64_t *)scratch;
  a.err = err_flag;
  const int lists = (int)((rel_end - rel_begin + k - 1) / k);
  a.key_row = (int64_t)lists * k;
  KGE_CUDA_OK(cudaMemsetAsync(scratch, 0, need, st));   // key 0 for the excluded relations and the padding
  if ((rc = dispatch_relation<EPI_KEYS>(m->model, a, st))) return rc;
  return kge_eval_topk_merge(a.keys, Q, lists, k, keys_out, nullptr, nullptr, stream);
}

extern "C" int kge_eval_relation_filter_bits(const int64_t *index_keys, const int64_t *index_offsets,
                                             const int32_t *index_relations, int64_t nkeys, const int64_t *queries,
                                             int64_t Q, int64_t nentity, int64_t nrelation, uint32_t *bits,
                                             void *stream) {
  KGE_REQUIRE(bits && (queries || Q == 0) && Q >= 0 && nentity > 0 && nrelation > 0 && nkeys >= 0, "bad arguments");
  KGE_REQUIRE(nkeys == 0 || (index_keys && index_offsets && index_relations), "null filter index");
  if (Q == 0) return KGE_OK;
  const int words = (int)((nrelation + 31) / 32);
  cudaStream_t st = (cudaStream_t)stream;
  KGE_CUDA_OK(cudaMemsetAsync(bits, 0, sizeof(uint32_t) * (size_t)Q * words, st));
  if (nkeys == 0) return KGE_OK;
  const int grid = (int)((Q + 127) / 128 < 148 * 4 ? (Q + 127) / 128 : 148 * 4);
  relation_lookup_kernel<<<grid, 128, 0, st>>>(index_keys, index_offsets, index_relations, nkeys, queries, Q, nentity,
                                               nrelation, words, bits);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}
