// kge_eval_path.cu -- path queries (a, r1/r2/.../rL, ?) (Guu et al. 2015, "Traversing Knowledge Graphs in Vector Space").
//
// A path query is scored by folding its hops into one query vector q and ranking every entity against q with the
// one-hop kernels of kge_eval.cu / kge_eval_gemm.cu / kge_eval_topk.cu, which read nothing but q, the positive column of
// `queries` and a [Q, ceil(nentity/32)] bitmap.  This file makes the two inputs those kernels cannot:
//   path_query_vectors  the fold of an L-hop path into q, with the non-contracted primitives of build_q, so that a one-hop
//                       forward path gives build_q's vector bit for bit (DESIGN.md section 3.13)
//   path_hop            one hop of the answer-set traversal: the frontier bitmap of every query mapped through the resident
//                       filter index into the next bitmap (ping-pong, one launch per hop); the last one is the filter
//                       bitmap of the count / top-k kernels, in the filter_bits layout
// Hop ids: r in [0, nrelation) follows relation r, r + nrelation follows it inverted, -1 pads a row after its last hop.
#include "kge_eval_tile.cuh"

namespace kge {

// ---- the fold ----------------------------------------------------------------------------------------------------
// One element k of q through one hop.  ComplEx / RotatE take build_q's tail formula (q * r) or head formula (q * conj r)
// with F = q; which one follows from the mode and the hop's direction.
template <int MODEL, bool HEAD>
__device__ __forceinline__ void path_hop_element(float &q0, float &q1, const float *__restrict__ Rr, int k, int d,
                                                 float scale, bool inv) {
  if constexpr (MODEL == KGE_TRANSE) {
    const float r = Rr[k];
    q0 = inv ? fsub(q0, r) : (HEAD ? fadd(r, q0) : fadd(q0, r));
  } else if constexpr (MODEL == KGE_DISTMULT) {
    const float r = Rr[k];
    q0 = HEAD ? fmul(r, q0) : fmul(q0, r);
  } else if constexpr (MODEL == KGE_COMPLEX || MODEL == KGE_ROTATE) {
    float rr, ri;
    if constexpr (MODEL == KGE_COMPLEX) {
      rr = Rr[k];
      ri = Rr[d + k];
    } else {
      sincos_rep(fdiv(Rr[k], scale), &ri, &rr);
    }
    if (HEAD == inv) {                                      // tail formula: q * r
      const float n0 = fsub(fmul(q0, rr), fmul(q1, ri));
      q1 = fadd(fmul(q0, ri), fmul(q1, rr));
      q0 = n0;
    } else {                                                // head formula: conj(r) * q
      const float n0 = fadd(fmul(rr, q0), fmul(ri, q1));
      q1 = fsub(fmul(rr, q1), fmul(ri, q0));
      q0 = n0;
    }
  } else {                                                  // pRotatE: phases add
    const float pr = fdiv(Rr[k], scale);
    q0 = inv ? fsub(q0, pr) : (HEAD ? fadd(pr, q0) : fadd(q0, pr));
  }
}

// One CTA per query.  Tail-batch applies hops 1..L to row(a); head-batch starts from row(a) (negated for TransE and
// pRotatE, whose one-hop head query is r - t) and applies hops L..1.  A bad anchor, hop id or padding sets *err and folds
// a zero row.
template <int MODEL, bool HEAD>
__global__ void __launch_bounds__(128) path_query_vectors_kernel(const float *__restrict__ E, const float *__restrict__ R,
                                                                 const int64_t *__restrict__ anchors,
                                                                 const int64_t *__restrict__ paths, int64_t Q, int64_t L,
                                                                 int64_t nentity, int64_t nrelation, int d, int De,
                                                                 int Dr, float scale, float *__restrict__ qvec,
                                                                 int32_t *err) {
  constexpr bool CPLX = MODEL == KGE_COMPLEX || MODEL == KGE_ROTATE;
  for (int64_t qi = blockIdx.x; qi < Q; qi += gridDim.x) {
    const int64_t *row = paths + qi * L;
    const int64_t a = anchors[qi];
    bool ok = (uint64_t)a < (uint64_t)nentity;
    int64_t len = 0;
    while (len < L && row[len] != -1) ok &= (uint64_t)row[len++] < (uint64_t)(2 * nrelation);
    for (int64_t s = len; s < L; ++s) ok &= row[s] == -1;   // padding only after the last hop
    ok &= len >= 1;
    float *q = qvec + qi * De;
    if (!ok) {
      if (threadIdx.x == 0 && err) *err = 1;
      for (int k = threadIdx.x; k < De; k += blockDim.x) q[k] = 0.f;
      continue;
    }
    const float *A = E + a * De;
    for (int k = threadIdx.x; k < d; k += blockDim.x) {
      float q0 = A[k], q1 = CPLX ? A[d + k] : 0.f;
      if constexpr (MODEL == KGE_PROTATE) q0 = fdiv(q0, scale);
      if constexpr (HEAD && (MODEL == KGE_TRANSE || MODEL == KGE_PROTATE)) q0 = -q0;
      for (int64_t t = 0; t < len; ++t) {
        const int64_t h = row[HEAD ? len - 1 - t : t];
        const bool inv = h >= nrelation;
        path_hop_element<MODEL, HEAD>(q0, q1, R + (inv ? h - nrelation : h) * Dr, k, d, scale, inv);
      }
      q[k] = q0;
      if constexpr (CPLX) q[d + k] = q1;
    }
  }
}

// ---- the traversal -----------------------------------------------------------------------------------------------
// The two layouts of the resident filter index (model.py _filter_tables).  run(key) gives the run [b, e) of the key's
// entities; a null index finds nothing.
struct DenseIndex {                  // direct-address CSR of kge_eval_filter_index_build: two loads per lookup
  const int32_t *offsets, *entities;
  __device__ __forceinline__ void run(int64_t key, int64_t &b, int64_t &e) const {
    if (offsets) { b = offsets[key]; e = offsets[key + 1]; }
  }
};
struct SortedIndex {                 // host-built sorted-key CSR (FilterIndex.table): binary search
  const int64_t *keys, *offsets;
  const int32_t *entities;
  int64_t nkeys;
  __device__ __forceinline__ void run(int64_t key, int64_t &b, int64_t &e) const {
    int64_t lo = 0, hi = nkeys;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (lo < nkeys && keys[lo] == key) { b = offsets[lo]; e = offsets[lo + 1]; }
  }
};

__global__ void path_seed_kernel(const int64_t *__restrict__ anchors, int64_t Q, int64_t nentity, int words,
                                 uint32_t *__restrict__ bits) {
  for (int64_t qi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; qi < Q; qi += (int64_t)gridDim.x * blockDim.x) {
    const int64_t a = anchors[qi];
    if ((uint64_t)a < (uint64_t)nentity) bits[qi * words + (a >> 5)] = 1u << (a & 31);
  }
}

// Hop `step` of every query: next = union over the entities e set in cur of the run of e's key.  One warp per (query,
// 32 words): each lane takes the set bits of its word one at a time and looks its run up, then the warp strides every
// non-empty run of the round together with atomicOr, so a hub with tens of thousands of neighbours is spread over the
// lanes.  Tail-batch takes hop `step`, head-batch hop len-1-step; a query with fewer hops copies its frontier.  Forward
// tail hops and inverse head hops read the tail index ((e, r) -> tails), the other two the head index ((r, e) -> heads).
template <class Index>
__global__ void path_hop_kernel(const Index tail_ix, const Index head_ix, const int64_t *__restrict__ paths, int64_t Q,
                                int64_t L, int64_t step, int head_batch, int64_t nentity, int64_t nrelation, int words,
                                const uint32_t *__restrict__ cur, uint32_t *__restrict__ nxt) {
  const int lane = threadIdx.x & 31;
  const unsigned groups = (unsigned)(words + 31) / 32, tasks = (unsigned)Q * groups;      // < 2^31 (path_bits)
  const unsigned nwarps = (gridDim.x * blockDim.x) >> 5;
  for (unsigned task = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; task < tasks; task += nwarps) {
    const int64_t qi = task / groups;                                                   // (32-bit division: no call)
    const int w = (int)(task - (unsigned)qi * groups) * 32 + lane;
    const int64_t *row = paths + qi * L;
    int64_t len = 0;
    while (len < L && row[len] >= 0) ++len;
    uint32_t word = w < words ? cur[qi * words + w] : 0u;
    uint32_t *out = nxt + qi * words;
    if (step >= len) {                                      // path already ended: carry the frontier
      if (w < words) out[w] = word;
      continue;
    }
    const int64_t h = row[head_batch ? len - 1 - step : step];
    if (h >= 2 * nrelation) continue;                       // bad hop id (flagged by the fold): nothing is reached
    const bool inv = h >= nrelation;
    const int64_t r = inv ? h - nrelation : h;
    const bool tail = head_batch ? inv : !inv;
    const Index ix = tail ? tail_ix : head_ix;
    while (__any_sync(0xffffffffu, word != 0u)) {
      int64_t b = 0, e = 0;
      if (word) {
        const int64_t ent = (int64_t)w * 32 + (__ffs(word) - 1);
        word &= word - 1;
        ix.run(tail ? ent * nrelation + r : r * nentity + ent, b, e);
      }
      for (uint32_t pending = __ballot_sync(0xffffffffu, e > b); pending; pending &= pending - 1) {
        const int l = __ffs(pending) - 1;
        const int64_t rb = __shfl_sync(0xffffffffu, b, l), re = __shfl_sync(0xffffffffu, e, l);
        for (int64_t i = rb + lane; i < re; i += 32) {
          const int32_t j = ix.entities[i];
          if (j >= 0 && j < nentity) atomicOr(out + (j >> 5), 1u << (j & 31));
        }
      }
    }
  }
}

// answer_counts[q] = popcount of the query's final bitmap, one warp per query
__global__ void path_count_kernel(const uint32_t *__restrict__ bits, int64_t Q, int words, int32_t *__restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t qi = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; qi < Q; qi += nwarps) {
    int c = 0;
    for (int w = lane; w < words; w += 32) c += __popc(bits[qi * words + w]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) counts[qi] = c;
  }
}

template <class Index>
static int path_bits(const Index &tail_ix, const Index &head_ix, const int64_t *anchors, const int64_t *paths, int64_t Q,
                     int64_t L, int mode, int64_t nentity, int64_t nrelation, uint32_t *bits, uint32_t *pong,
                     int32_t *answer_counts, void *stream) {
  const int words = (int)((nentity + 31) / 32);
  const size_t bytes = sizeof(uint32_t) * (size_t)Q * words;
  cudaStream_t st = (cudaStream_t)stream;
  uint32_t *cur = L % 2 ? pong : bits, *nxt = L % 2 ? bits : pong;      // the last hop writes `bits`
  KGE_CUDA_OK(cudaMemsetAsync(cur, 0, bytes, st));
  path_seed_kernel<<<(int)((Q + 255) / 256 < 148 * 8 ? (Q + 255) / 256 : 148 * 8), 256, 0, st>>>(anchors, Q, nentity,
                                                                                                words, cur);
  KGE_CUDA_OK(cudaGetLastError());
  const int64_t warps = Q * ((words + 31) / 32);
  KGE_REQUIRE(warps < (1ll << 31), "%lld queries x %d bitmap words are too many for one call", (long long)Q, words);
  const int grid = (int)((warps + 7) / 8 < 148 * 16 ? (warps + 7) / 8 : 148 * 16);
  for (int64_t step = 0; step < L; ++step) {
    KGE_CUDA_OK(cudaMemsetAsync(nxt, 0, bytes, st));
    path_hop_kernel<Index><<<grid, 256, 0, st>>>(tail_ix, head_ix, paths, Q, L, step, mode == KGE_HEAD_BATCH, nentity,
                                                 nrelation, words, cur, nxt);
    KGE_CUDA_OK(cudaGetLastError());
    uint32_t *t = cur; cur = nxt; nxt = t;
  }
  if (answer_counts) {
    path_count_kernel<<<(int)((Q + 7) / 8 < 148 * 16 ? (Q + 7) / 8 : 148 * 16), 256, 0, st>>>(bits, Q, words,
                                                                                               answer_counts);
    KGE_CUDA_OK(cudaGetLastError());
  }
  return KGE_OK;
}

static int path_bits_args(const int64_t *anchors, const int64_t *paths, int64_t Q, int64_t L, int mode, int64_t nentity,
                          int64_t nrelation, const uint32_t *bits, const uint32_t *pong) {
  KGE_REQUIRE(mode == KGE_HEAD_BATCH || mode == KGE_TAIL_BATCH, "negative batch mode %d not supported", mode);
  KGE_REQUIRE(Q >= 0 && nentity > 0 && nrelation > 0, "bad arguments");
  KGE_REQUIRE(L >= 1, "a path has at least one hop, got L = %lld", (long long)L);
  KGE_REQUIRE((anchors && paths && bits && pong) || Q == 0, "null pointer");
  KGE_REQUIRE(bits != pong || Q == 0, "bits and pong must be two buffers");
  return KGE_OK;
}

}  // namespace kge

using namespace kge;

extern "C" int kge_eval_path_query_vectors(const kge_model_t *m, int mode, const int64_t *anchors, const int64_t *paths,
                                           int64_t Q, int64_t L, float *qvec, int32_t *err_flag, void *stream) {
  int rc = check_model(m);
  if (rc) return rc;
  bool head;
  if ((rc = eval_mode(mode, head))) return rc;
  KGE_REQUIRE(Q >= 0, "bad query count %lld", (long long)Q);
  KGE_REQUIRE(L >= 1, "a path has at least one hop, got L = %lld", (long long)L);
  KGE_REQUIRE((anchors && paths && qvec) || Q == 0, "null pointer");
  if (Q == 0) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  const bool cplx = m->model == KGE_COMPLEX || m->model == KGE_ROTATE;
  const int d = cplx ? (int)(m->entity_dim / 2) : (int)m->entity_dim;
  const int grid = (int)(Q < 148 * 16 ? Q : 148 * 16);
  const float scale = phase_scale(m);
  cudaStream_t st = (cudaStream_t)stream;
#define KGE_PQV(MODEL)                                                                                                 \
  case MODEL:                                                                                                          \
    if (head)                                                                                                          \
      path_query_vectors_kernel<MODEL, true><<<grid, 128, 0, st>>>(m->entity, m->relation, anchors, paths, Q, L,       \
                                                                   m->nentity, m->nrelation, d, (int)m->entity_dim,    \
                                                                   (int)m->relation_dim, scale, qvec, err_flag);       \
    else                                                                                                               \
      path_query_vectors_kernel<MODEL, false><<<grid, 128, 0, st>>>(m->entity, m->relation, anchors, paths, Q, L,      \
                                                                    m->nentity, m->nrelation, d, (int)m->entity_dim,   \
                                                                    (int)m->relation_dim, scale, qvec, err_flag);      \
    break;
  switch (m->model) {
    KGE_PQV(KGE_TRANSE)
    KGE_PQV(KGE_DISTMULT)
    KGE_PQV(KGE_COMPLEX)
    KGE_PQV(KGE_ROTATE)
    KGE_PQV(KGE_PROTATE)
  }
#undef KGE_PQV
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

extern "C" int kge_eval_path_bits_dense(const int32_t *tail_offsets, const int32_t *tail_entities,
                                        const int32_t *head_offsets, const int32_t *head_entities, const int64_t *anchors,
                                        const int64_t *paths, int64_t Q, int64_t L, int mode, int64_t nentity,
                                        int64_t nrelation, uint32_t *bits, uint32_t *pong, int32_t *answer_counts,
                                        void *stream) {
  int rc = path_bits_args(anchors, paths, Q, L, mode, nentity, nrelation, bits, pong);
  if (rc) return rc;
  KGE_REQUIRE(!tail_offsets == !tail_entities && !head_offsets == !head_entities, "half of a filter index is null");
  KGE_REQUIRE(nentity * nrelation < (1ll << 31) - 1024, "key space of %lld entries is too large for the direct-address index",
              (long long)(nentity * nrelation));
  if (Q == 0) return KGE_OK;
  return path_bits(DenseIndex{tail_offsets, tail_entities}, DenseIndex{head_offsets, head_entities}, anchors, paths, Q, L,
                   mode, nentity, nrelation, bits, pong, answer_counts, stream);
}

extern "C" int kge_eval_path_bits(const int64_t *tail_keys, const int64_t *tail_offsets, const int32_t *tail_entities,
                                  int64_t tail_nkeys, const int64_t *head_keys, const int64_t *head_offsets,
                                  const int32_t *head_entities, int64_t head_nkeys, const int64_t *anchors,
                                  const int64_t *paths, int64_t Q, int64_t L, int mode, int64_t nentity, int64_t nrelation,
                                  uint32_t *bits, uint32_t *pong, int32_t *answer_counts, void *stream) {
  int rc = path_bits_args(anchors, paths, Q, L, mode, nentity, nrelation, bits, pong);
  if (rc) return rc;
  KGE_REQUIRE(tail_nkeys >= 0 && head_nkeys >= 0, "bad arguments");
  KGE_REQUIRE((tail_nkeys == 0 || (tail_keys && tail_offsets && tail_entities)) &&
                  (head_nkeys == 0 || (head_keys && head_offsets && head_entities)),
              "null filter index");
  if (Q == 0) return KGE_OK;
  return path_bits(SortedIndex{tail_keys, tail_offsets, tail_entities, tail_nkeys},
                   SortedIndex{head_keys, head_offsets, head_entities, head_nkeys}, anchors, paths, Q, L, mode, nentity,
                   nrelation, bits, pong, answer_counts, stream);
}
