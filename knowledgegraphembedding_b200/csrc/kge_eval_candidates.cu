// kge_eval_candidates.cu -- rank statistics of each query against its own list of candidate entities (the sampled
// evaluation protocol: KGEModel.candidate_rank_statistics).
//
// The lists of two queries share no rows, so there is no [queries x entities] tile to reuse a row across: the kernel
// gathers rows instead.  One CTA scores CAND_THREADS listed entries of one query, one lane per entry:
//   * the query vector is staged once per CTA in shared memory and read by every lane at the same address (broadcast);
//   * the listed rows are staged SK floats (per complex half) at a time by a double-buffered cp.async ring, 4 lanes per
//     64-byte row segment, at a row stride of SST = SK + 4 floats, so that the 16-byte reads of 8 consecutive lanes
//     fall on 8 distinct bank groups (SST / 4 is odd);
//   * every lane sums its own row in the canonical order of kge_eval_tile.cuh (blocks of KC = 32 consecutive k, each
//     summed in index order from 0.0f, block sums added in index order) with the same op_exact, so every score is the
//     bit pattern of the all-entity kernels and of the C oracle;
//   * the six counters go through per-CTA shared counters (a warp reduction first) and one global atomic per counter.
// All lanes are busy at every width: a lane owns a pair, not a 32-wide block of one pair (the warp-per-pair mapping of
// canonical_pair_score leaves 28 of 32 lanes idle at d = 100).
#include "kge_eval_tile.cuh"

namespace kge {

constexpr int CAND_THREADS = 128;          // listed entries per CTA
constexpr int SK = 16, SST = SK + 4;       // staged k per ring stage (half a canonical block) and the row stride
static_assert(KC % SK == 0 && (SST / 4) % 2 == 1, "stages tile the canonical blocks; conflict-free 16-byte reads");

struct CandArgs {
  const float *qvec;            // [Q, De]
  const float *X;               // candidate table [nentity, De] (entity table, or phase table for pRotatE)
  const int64_t *queries;       // [Q, 3]
  const float *pos_score;       // [Q]
  const int64_t *cand;          // [Q, ld] entity ids, -1 = padding
  const uint32_t *filter_bits;  // [Q, words] or null
  int32_t *stats;               // [Q, KGE_RANK_STATS]
  float *scores_out;            // [Q, ld] or null
  int32_t *err;
  const float *modulus;
  int64_t nentity, ld, col_begin, col_end;
  int d, De, dq, pos_col, words;
  float gamma;
};

// Stage k in [k0, k0 + SK) of both halves of every listed row of the CTA into one ring slot: plane h, row r at
// slot + (h * CAND_THREADS + r) * SST.  Entries past d and padding rows are left unwritten: no lane reads them.
template <bool CPLX, bool ALIGNED>
__device__ __forceinline__ void stage_rows(const CandArgs &a, const int64_t *ids, float *slot, int k0) {
  constexpr int H = CPLX ? 2 : 1, VPR = SK / 4;
  for (int idx = threadIdx.x; idx < CAND_THREADS * H * VPR; idx += CAND_THREADS) {
    const int v = idx % VPR, h = (idx / VPR) % H, row = idx / (VPR * H);
    const int k = k0 + 4 * v;
    const int64_t g = ids[row];
    if (g < 0 || k >= a.d) continue;
    const float *src = a.X + g * a.De + h * a.d + k;
    float *dst = slot + (h * CAND_THREADS + row) * SST + 4 * v;
    if constexpr (ALIGNED) {
      cp_async16(dst, src, true);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) dst[e] = (k + e < a.d) ? src[e] : 0.f;
    }
  }
}

template <int OP>
__device__ __forceinline__ float add4(float part, const float *q, const float *x, int qoff, int xoff) {
  constexpr bool CPLX = op_is_complex(OP);
  const float4 qa = *reinterpret_cast<const float4 *>(q), xa = *reinterpret_cast<const float4 *>(x);
  float4 qb = make_float4(0.f, 0.f, 0.f, 0.f), xb = qb;
  if constexpr (CPLX) {
    qb = *reinterpret_cast<const float4 *>(q + qoff);
    xb = *reinterpret_cast<const float4 *>(x + xoff);
  }
  part = fadd(part, op_exact<OP>(qa.x, qb.x, xa.x, xb.x));
  part = fadd(part, op_exact<OP>(qa.y, qb.y, xa.y, xb.y));
  part = fadd(part, op_exact<OP>(qa.z, qb.z, xa.z, xb.z));
  part = fadd(part, op_exact<OP>(qa.w, qb.w, xa.w, xb.w));
  return part;
}

// grid (Q, column tiles): CTA (q, t) scores the entries [col_begin + t * CAND_THREADS, ...) of query q's list.
template <int OP, bool ALIGNED>
__global__ void __launch_bounds__(CAND_THREADS) candidate_stats_kernel(const CandArgs a) {
  constexpr bool CPLX = op_is_complex(OP);
  constexpr int H = CPLX ? 2 : 1;
  constexpr int SLOT = H * CAND_THREADS * SST;
  extern __shared__ __align__(16) float smem[];
  float *sq = smem + 2 * SLOT;                             // [H][dq]: the query vector, zero in [d, dq)
  __shared__ int64_t ids[CAND_THREADS];
  __shared__ int cnt[KGE_RANK_STATS];

  const int tid = threadIdx.x;
  const int64_t qi = blockIdx.x;
  const int64_t col = a.col_begin + (int64_t)blockIdx.y * CAND_THREADS + tid;
  int64_t id = -1;
  if (col < a.col_end) {
    id = a.cand[qi * a.ld + col];
    if (id < -1 || id >= a.nentity) {                      // not an entity and not padding
      *a.err = 1;
      id = -1;
    }
  }
  ids[tid] = id;
  if (tid < KGE_RANK_STATS) cnt[tid] = 0;
  for (int i = tid; i < H * a.dq; i += CAND_THREADS) {
    const int h = i / a.dq, k = i - h * a.dq;
    sq[i] = k < a.d ? a.qvec[qi * a.De + h * a.d + k] : 0.f;
  }
  __syncthreads();

  const int nst = (a.d + SK - 1) / SK;
  stage_rows<CPLX, ALIGNED>(a, ids, smem, 0);
  cp_async_commit();
  float acc = 0.f, part = 0.f;
  for (int c = 0; c < nst; ++c) {
    if (c + 1 < nst) stage_rows<CPLX, ALIGNED>(a, ids, smem + ((c + 1) & 1) * SLOT, (c + 1) * SK);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const int k0 = c * SK;
    const float *x = smem + (c & 1) * SLOT + tid * SST;
    const float *q = sq + k0;
    if (k0 % KC == 0) part = 0.f;                          // a canonical block starts
    const int klen = a.d - k0 < SK ? a.d - k0 : SK;        // entries beyond d within a float4 are zero in q and x
    if (klen == SK) {
#pragma unroll
      for (int kk = 0; kk < SK; kk += 4) part = add4<OP>(part, q + kk, x + kk, a.dq, CAND_THREADS * SST);
    } else {
      for (int kk = 0; kk < klen; kk += 4) part = add4<OP>(part, q + kk, x + kk, a.dq, CAND_THREADS * SST);
    }
    if ((k0 + SK) % KC == 0 || c + 1 == nst) acc = fadd(acc, part);
    __syncthreads();
  }

  const float s = finish_exact<OP>(acc, a.gamma, a.modulus ? a.modulus[0] : 1.f);
  const float sp = a.pos_score[qi];
  const int64_t pid = a.queries[qi * 3 + a.pos_col];
  int c[KGE_RANK_STATS] = {0, 0, 0, 0, 0, 0};
  if (id >= 0 && id != pid) {                              // NaN is never greater or equal; -0.0 == +0.0
    const bool kept = !a.filter_bits || !((a.filter_bits[qi * a.words + (id >> 5)] >> (id & 31)) & 1u);
    const bool gt = s > sp, eb = s == sp && id < pid, ea = s == sp && id > pid;
    c[0] = kept && gt;
    c[1] = kept && eb;
    c[2] = kept && ea;
    c[3] = gt;
    c[4] = eb;
    c[5] = ea;
  }
  if (a.scores_out && col < a.col_end) a.scores_out[qi * a.ld + col] = id < 0 ? -INFINITY : id == pid ? sp : s;
#pragma unroll
  for (int k = 0; k < KGE_RANK_STATS; ++k) {
    const int w = __reduce_add_sync(0xffffffffu, c[k]);
    if ((tid & 31) == 0 && w) atomicAdd(&cnt[k], w);
  }
  __syncthreads();
  if (tid < KGE_RANK_STATS && cnt[tid]) atomicAdd(&a.stats[qi * KGE_RANK_STATS + tid], cnt[tid]);
}

template <int OP>
static int launch_candidates(const CandArgs &a, bool aligned, int64_t Q, cudaStream_t st) {
  constexpr int H = op_is_complex(OP) ? 2 : 1;
  const size_t smem = sizeof(float) * ((size_t)2 * H * CAND_THREADS * SST + (size_t)H * a.dq);
  const dim3 grid((unsigned)Q, (unsigned)((a.col_end - a.col_begin + CAND_THREADS - 1) / CAND_THREADS));
  auto k = aligned ? candidate_stats_kernel<OP, true> : candidate_stats_kernel<OP, false>;
  KGE_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<grid, CAND_THREADS, smem, st>>>(a);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

}  // namespace kge

using namespace kge;

extern "C" int kge_eval_candidate_rank_stats(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                                             int64_t Q, const float *phase_table, const float *pos_score,
                                             const int64_t *candidates, int64_t ld, int64_t col_begin, int64_t col_end,
                                             const uint32_t *filter_bits, int32_t *stats, float *scores_out,
                                             int32_t *err_flag, void *stream) {
  int rc = check_model(m);
  if (rc) return rc;
  bool head;
  if ((rc = eval_mode(mode, head))) return rc;
  KGE_REQUIRE(qvec && queries && pos_score && candidates && stats && err_flag, "null pointer");
  KGE_REQUIRE(Q >= 0, "negative query count %lld", (long long)Q);
  KGE_REQUIRE(ld >= 1, "candidate row length %lld must be at least 1", (long long)ld);
  KGE_REQUIRE(col_begin >= 0 && col_begin <= col_end && col_end <= ld, "column slice [%lld,%lld) outside [0,%lld)",
              (long long)col_begin, (long long)col_end, (long long)ld);
  if (Q == 0 || col_begin == col_end) return KGE_OK;
  KGE_REQUIRE(Q <= 0x7fffffff && (col_end - col_begin + CAND_THREADS - 1) / CAND_THREADS <= 65535,
              "at most 2^31-1 queries and %d columns per call", 65535 * CAND_THREADS);
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  EvalArgs e{};
  if ((rc = fill_eval_args(m, head, qvec, queries, Q, phase_table, e))) return rc;
  CandArgs a{};
  a.qvec = e.qvec; a.X = e.X; a.queries = queries; a.pos_score = pos_score; a.cand = candidates;
  a.filter_bits = filter_bits; a.stats = stats; a.scores_out = scores_out; a.err = err_flag; a.modulus = e.modulus;
  a.nentity = e.nentity; a.ld = ld; a.col_begin = col_begin; a.col_end = col_end;
  a.d = e.d; a.De = e.De; a.dq = (e.d + SK - 1) / SK * SK; a.pos_col = e.pos_col; a.words = e.words; a.gamma = e.gamma;
  const bool aligned = eval_aligned(e);
  cudaStream_t st = (cudaStream_t)stream;
#define KGE_CC(OP) \
  case OP:         \
    return launch_candidates<OP>(a, aligned, Q, st);
  switch (op_of(m->model, head)) {
    KGE_CC(OP_SUBABS) KGE_CC(OP_ADDABS) KGE_CC(OP_MUL) KGE_CC(OP_CMUL) KGE_CC(OP_CDIST) KGE_CC(OP_SUBSIN)
    KGE_CC(OP_ADDSIN)
  }
#undef KGE_CC
  set_error("unreachable");
  return KGE_ERR_INVALID;
}
