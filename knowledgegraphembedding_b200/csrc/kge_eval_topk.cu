// kge_eval_topk.cu -- top-k link prediction: the k best entities of every query (h, r, ?) / (?, r, t), fused into the
// canonical score tiles so that the [Q, nentity] score matrix never exists.
//
//   topk_kernel        grid (entity strips x query tiles of 64).  A CTA runs tile_mainloop (kge_eval_tile.cuh: the
//                      scores are bit-identical to count_ranks_kernel's and oracle/kge_oracle.c's) over the 64-entity
//                      tiles of its strip and keeps, per query, a sorted list of its k best keys in shared memory;
//                      after each tile only the candidates above a query's current k-th key are merged in.
//   topk_merge_kernel  one CTA per query: radix-selects the k best of `lists` sorted lists (the strips of one call, or
//                      the entity shards of the ranks), sorts them and decodes ids / scores.
//
// Similarity search (kge_similarity_*) runs the same topk_kernel on the rows of one table: the query vectors are table
// rows (gather_rows_kernel) or free vectors, the element op is that of the metric (dot, cosine: OP_MUL; l1: OP_SUBABS;
// l2: OP_SQDIFF), the sum is canonical, and finish_sim turns it into a "larger is more similar" score; cosine also reads
// the row norms of row_norms_kernel.
//
// Order: score descending, then entity id ascending (the tie rule of the filtered rank); NaN after every number; -0.0
// and +0.0 are one value.  A candidate is one uint64 key, (orderable(score) << 32) | (0xFFFFFFFF - id): a larger key
// is a better candidate, and key 0 (no entity has id 0xFFFFFFFF) marks an empty slot.
#include "kge_eval_tile.cuh"

namespace kge {

__device__ __forceinline__ void topk_decode(uint64_t key, int64_t &id, float &score) {
  if (key == 0) {
    id = -1;
    score = __uint_as_float(0xFF800000u);                  // -inf
    return;
  }
  const uint32_t ord = (uint32_t)(key >> 32);
  id = (int64_t)(0xFFFFFFFFu - (uint32_t)key);
  score = ord == 0 ? __uint_as_float(0x7FC00000u) : __uint_as_float((ord & 0x80000000u) ? (ord & 0x7FFFFFFFu) : ~ord);
}

struct TopkArgs {
  const uint32_t *exclude;      // [Q, words] or null
  uint64_t *lists;              // [Q, strips, k]
  int k, strips, tiles_per_strip;
  const float *qnorm, *xnorm;   // similarity, cosine: norms of the query vectors [Q] and of the table rows [rows]
  const int64_t *self_ids;      // similarity: [Q] row left out of each query's list (-1: none), or null
};

// What a topk_kernel instantiation selects on: link prediction (SIM_LINK: finish_exact<OP>, the exclusion bitmap) or a
// similarity metric KGE_SIM_* (finish_sim<SIM>, the query's own row left out).  Scores are "larger is more similar".
constexpr int SIM_LINK = -1;
template <int SIM>
__device__ __forceinline__ float finish_sim(float acc, float qnorm, float xnorm) {
  if constexpr (SIM == KGE_SIM_DOT) return acc;
  else if constexpr (SIM == KGE_SIM_COSINE) return fdiv(acc, fmul(qnorm, xnorm));       // a zero row: 0/0 = NaN, last
  else if constexpr (SIM == KGE_SIM_L2) return -fsqrt(acc);
  else return -acc;                                                                      // KGE_SIM_L1
}

constexpr int TOPK_CAND = TJ;   // candidates of one query per tile (one per entity of the tile)

// Shared memory: the two staging buffers of tile_mainloop (which also hold the candidates of a tile between the
// mainloop and the merge), then [TQ, k] keys; the thresholds and candidate counts are static.
template <int OP, bool ALIGNED, int SIM>
__global__ void __launch_bounds__(EVAL_THREADS, 2) topk_kernel(const EvalArgs a, const TopkArgs t) {
  constexpr int H = op_is_complex(OP) ? 2 : 1;
  constexpr int STAGING = 2 * (TQ + TJ) * H * ST;          // floats
  static_assert(STAGING * sizeof(float) >= TQ * TOPK_CAND * sizeof(uint64_t), "candidates alias the staging buffers");
  extern __shared__ __align__(16) float smem[];
  uint64_t *cand = reinterpret_cast<uint64_t *>(smem);
  uint64_t *list = reinterpret_cast<uint64_t *>(smem + STAGING);
  __shared__ uint64_t thr[TQ];
  __shared__ int ncand[TQ];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tq = tid % 16, tj = tid / 16;
  const int k = t.k;
  const int64_t q0 = (int64_t)blockIdx.y * TQ;
  const int strip = blockIdx.x;
  for (int i = tid; i < TQ * k; i += EVAL_THREADS) list[i] = 0;
  if (tid < TQ) {
    thr[tid] = 0;
    ncand[tid] = 0;
  }
  __syncthreads();
  const float modulus = a.modulus ? a.modulus[0] : 1.f;
  const int64_t ntiles = (a.ent_end - a.ent_begin + TJ - 1) / TJ;
  const int64_t tile_end = min((int64_t)(strip + 1) * t.tiles_per_strip, ntiles);

  for (int64_t tile = (int64_t)strip * t.tiles_per_strip; tile < tile_end; ++tile) {
    const int64_t j0 = a.ent_begin + tile * TJ;
    const TileAcc acc = tile_mainloop<OP, ALIGNED>(a, smem, q0, j0, tq, tj);

    // ---- candidates above the query's current k-th key (the staging buffers are free until the next tile) ----------
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int ql = tq + 16 * i;
      const int64_t qi = q0 + ql;
      if (qi >= a.Q) continue;
      const uint64_t bar = thr[ql];
      const uint32_t *ex = SIM == SIM_LINK && t.exclude ? t.exclude + qi * a.words : nullptr;
      int64_t self = -1;
      float qn = 0.f;
      if constexpr (SIM != SIM_LINK) {
        if (t.self_ids) self = t.self_ids[qi];
        if constexpr (SIM == KGE_SIM_COSINE) qn = t.qnorm[qi];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t ej = j0 + tj + 16 * j;
        if (ej >= a.ent_end) continue;
        float s;
        if constexpr (SIM == SIM_LINK) {
          if (ex && ((ex[ej >> 5] >> (ej & 31)) & 1u)) continue;
          s = finish_exact<OP>(acc.v[i][j], a.gamma, modulus);
        } else {
          if (ej == self) continue;
          s = finish_sim<SIM>(acc.v[i][j], qn, SIM == KGE_SIM_COSINE ? t.xnorm[ej] : 0.f);
        }
        const uint64_t key = topk_key(s, ej);
        if (key > bar) cand[ql * TOPK_CAND + atomicAdd(&ncand[ql], 1)] = key;
      }
    }
    __syncthreads();

    // ---- merge: one warp per query.  Keys are distinct, so the new position of a key is the number of keys of both
    // sets above it; positions >= k drop out.  Every candidate is above the list's k-th key. -------------------------
    for (int ql = warp; ql < TQ; ql += EVAL_THREADS / 32) {
      const int c = ncand[ql];
      if (c == 0) continue;
      uint64_t *L = list + ql * k;
      const uint64_t *C = cand + ql * TOPK_CAND;
      uint64_t lv[KGE_TOPK_MAX / 32], cv[TOPK_CAND / 32];
      int lp[KGE_TOPK_MAX / 32], cp[TOPK_CAND / 32];
#pragma unroll
      for (int u = 0; u < KGE_TOPK_MAX / 32; ++u) {
        const int idx = lane + 32 * u;
        lv[u] = idx < k ? L[idx] : 0;
        lp[u] = idx;
      }
#pragma unroll
      for (int u = 0; u < TOPK_CAND / 32; ++u) {
        const int idx = lane + 32 * u;
        cv[u] = idx < c ? C[idx] : 0;
        int lo = 0, hi = k;                                // list keys above cv[u] (the list is descending)
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (L[mid] > cv[u]) lo = mid + 1;
          else hi = mid;
        }
        cp[u] = lo;
      }
      for (int i = 0; i < c; ++i) {
        const uint64_t x = C[i];
#pragma unroll
        for (int u = 0; u < KGE_TOPK_MAX / 32; ++u) lp[u] += x > lv[u];
#pragma unroll
        for (int u = 0; u < TOPK_CAND / 32; ++u) cp[u] += x > cv[u];
      }
      __syncwarp();
#pragma unroll
      for (int u = 0; u < KGE_TOPK_MAX / 32; ++u)
        if (lane + 32 * u < k && lp[u] < k) L[lp[u]] = lv[u];
#pragma unroll
      for (int u = 0; u < TOPK_CAND / 32; ++u)
        if (lane + 32 * u < c && cp[u] < k) L[cp[u]] = cv[u];
      __syncwarp();
      if (lane == 0) {
        thr[ql] = L[k - 1];
        ncand[ql] = 0;
      }
    }
    __syncthreads();
  }

  // ---- this strip's list of every query of the tile --------------------------------------------------------------
  for (int i = tid; i < TQ * k; i += EVAL_THREADS) {
    const int ql = i / k, r = i - ql * k;
    const int64_t qi = q0 + ql;
    if (qi < a.Q) t.lists[(qi * t.strips + strip) * k + r] = list[i];
  }
}

// ---- k best of `lists` sorted key lists per query ------------------------------------------------------------------
constexpr int MERGE_THREADS = 256;
static_assert(MERGE_THREADS >= KGE_TOPK_MAX, "one thread per selected key");

__global__ void __launch_bounds__(MERGE_THREADS) topk_merge_kernel(const uint64_t *__restrict__ in, int64_t Q, int lists,
                                                                   int k, uint64_t *keys_out, int64_t *ids_out,
                                                                   float *scores_out) {
  __shared__ int hist[256];
  __shared__ uint64_t sel[KGE_TOPK_MAX];
  __shared__ uint64_t prefix_sh;
  __shared__ int remaining_sh, nsel;
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t n = (int64_t)lists * k;
  for (int64_t q = blockIdx.x; q < Q; q += gridDim.x) {
    const uint64_t *x = in + q * n;
    // MSB-first radix select of the k-th largest key T: after the 8 digits, `remaining` keys equal to T belong to the
    // top k (one at most, unless T is the empty key 0).
    uint64_t prefix = 0, mask = 0;
    int remaining = k;
    for (int shift = 56; shift >= 0; shift -= 8) {
      hist[tid] = 0;
      __syncthreads();
      for (int64_t i = tid; i < n; i += MERGE_THREADS) {
        const uint64_t v = x[i];
        if ((v & mask) == prefix) atomicAdd(&hist[(v >> shift) & 255], 1);
      }
      __syncthreads();
      if (tid < 32) {                                      // lane l holds bins 255 - 8l ... 248 - 8l (high bins first)
        int h[8], s = 0;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          h[b] = hist[255 - 8 * lane - b];
          s += h[b];
        }
        int incl = s;                                      // inclusive prefix over the lanes
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += y;
        }
        const int excl = incl - s;
        const unsigned hit = __ballot_sync(0xffffffffu, excl < remaining && remaining <= incl);
        if (lane == __ffs(hit) - 1) {
          int above = excl, b = 7;
          bool found = false;
#pragma unroll
          for (int bb = 0; bb < 8; ++bb) {                 // (unrolled: h[] stays in registers)
            if (found) continue;
            if (above + h[bb] >= remaining) {
              b = bb;
              found = true;
            } else {
              above += h[bb];
            }
          }
          prefix_sh = prefix | ((uint64_t)(255 - 8 * lane - b) << shift);
          remaining_sh = remaining - above;
        }
      }
      __syncthreads();
      prefix = prefix_sh;
      remaining = remaining_sh;
      mask |= (uint64_t)255 << shift;
    }
    const uint64_t T = prefix;
    if (tid == 0) nsel = 0;
    __syncthreads();
    for (int64_t i = tid; i < n; i += MERGE_THREADS) {
      const uint64_t v = x[i];
      if (v > T || (v == T && T != 0)) {
        const int slot = atomicAdd(&nsel, 1);
        if (slot < k) sel[slot] = v;                       // (more than k only if a caller passes duplicate keys)
      }
    }
    __syncthreads();
    const int ns = nsel < k ? nsel : k;
    if (tid < k) {
      int r = tid;
      uint64_t v = 0;
      if (tid < ns) {
        v = sel[tid];
        r = 0;
        for (int i = 0; i < ns; ++i) r += sel[i] > v;
      }
      if (keys_out) keys_out[q * k + r] = v;
      if (ids_out || scores_out) {
        int64_t id;
        float s;
        topk_decode(v, id, s);
        if (ids_out) ids_out[q * k + r] = id;
        if (scores_out) scores_out[q * k + r] = s;
      }
    }
    __syncthreads();
  }
}

// Strips: the CTAs of a launch run in waves of (SMs x CTAs per SM); a strip of w tiles costs w tile-times per wave, so the
// launch costs about ceil(CTAs / slots) * w.  Pick the strip count with the least such cost (fewest strips on a tie),
// at most 2048 / k strips so that the lists stay below 16 KB per query.
static int64_t topk_smem_bytes(bool cplx, int k) {
  return (int64_t)sizeof(float) * 2 * (TQ + TJ) * (cplx ? 2 : 1) * ST + (int64_t)sizeof(uint64_t) * TQ * k;
}
static int topk_strips(bool cplx, int64_t Q, int64_t nent, int k) {
  int64_t per_sm = (228 * 1024) / (topk_smem_bytes(cplx, k) + TQ * 12 + 1024);
  per_sm = per_sm < 1 ? 1 : per_sm > 2 ? 2 : per_sm;
  const int64_t slots = 148 * per_sm;
  const int64_t qtiles = (Q + TQ - 1) / TQ, ntiles = (nent + TJ - 1) / TJ;
  const int64_t max_strips = 2048 / k < ntiles ? (2048 / k < 1 ? 1 : 2048 / k) : ntiles;
  int64_t best = 1, best_cost = -1;
  for (int64_t s = 1; s <= max_strips; ++s) {
    const int64_t w = (ntiles + s - 1) / s, strips = (ntiles + w - 1) / w;     // no empty strip
    const int64_t cost = (qtiles * strips + slots - 1) / slots * w;
    if (best_cost < 0 || cost < best_cost) {
      best = strips;
      best_cost = cost;
    }
  }
  return (int)best;
}

static int topk_check(const kge_model_t *m, int64_t Q, int64_t ent_begin, int64_t ent_end, int k) {
  int rc = check_model(m);
  if (rc) return rc;
  KGE_REQUIRE(k >= 1 && k <= KGE_TOPK_MAX, "k = %d outside [1, %d]", k, KGE_TOPK_MAX);
  KGE_REQUIRE(Q >= 0 && (Q + TQ - 1) / TQ <= 65535, "at most %d queries per call", 65535 * TQ);
  KGE_REQUIRE(ent_begin >= 0 && ent_begin <= ent_end && ent_end <= m->nentity, "entity slice [%lld,%lld) outside [0,%lld)",
              (long long)ent_begin, (long long)ent_end, (long long)m->nentity);
  return KGE_OK;
}

static size_t topk_lists_bytes(const kge_model_t *m, int64_t Q, int64_t ent_begin, int64_t ent_end, int k) {
  if (Q == 0 || ent_begin == ent_end) return 0;
  const bool cplx = m->model == KGE_COMPLEX || m->model == KGE_ROTATE;
  return sizeof(uint64_t) * (size_t)Q * topk_strips(cplx, Q, ent_end - ent_begin, k) * k;
}

template <int OP, int SIM>
static int launch_topk(const EvalArgs &a, const TopkArgs &t, bool aligned, cudaStream_t st) {
  const size_t smem = (size_t)topk_smem_bytes(op_is_complex(OP), t.k);
  const dim3 grid((unsigned)t.strips, (unsigned)((a.Q + TQ - 1) / TQ));
  auto kern = aligned ? topk_kernel<OP, true, SIM> : topk_kernel<OP, false, SIM>;
  KGE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, EVAL_THREADS, smem, st>>>(a, t);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

static int launch_merge(const uint64_t *in, int64_t Q, int lists, int k, uint64_t *keys_out, int64_t *ids_out,
                        float *scores_out, cudaStream_t st) {
  const int grid = (int)(Q < 148 * 16 ? Q : 148 * 16);
  topk_merge_kernel<<<grid, MERGE_THREADS, 0, st>>>(in, Q, lists, k, keys_out, ids_out, scores_out);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

// ---- similarity search: query rows, row norms, argument checks ----------------------------------------------------
// rows_out[q] = X[ids[q]]; an id outside [0, rows) writes a zero row and sets *err (may be null).
constexpr int SIM_THREADS = 256;
__global__ void __launch_bounds__(SIM_THREADS) gather_rows_kernel(const float *__restrict__ X, int64_t rows, int width,
                                                                  const int64_t *__restrict__ ids, int64_t Q,
                                                                  float *__restrict__ rows_out, int32_t *err) {
  const int64_t n = Q * width;
  for (int64_t i = (int64_t)blockIdx.x * SIM_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * SIM_THREADS) {
    const int64_t q = i / width, c = i - q * width, id = ids[q];
    const bool ok = id >= 0 && id < rows;
    rows_out[i] = ok ? X[id * width + c] : 0.f;
    if (!ok && c == 0 && err) *err = 1;
  }
}

// out[r] = fsqrt(acc(X[r] . X[r])) in the canonical order (the sum topk_kernel forms for OP_MUL): one warp per row, lane
// l sums block b0 + l of KC elements in index order from +0.0f, then the block sums are added in index order.
__global__ void __launch_bounds__(SIM_THREADS) row_norms_kernel(const float *__restrict__ X, int64_t n, int width,
                                                                float *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (SIM_THREADS / 32) + (threadIdx.x >> 5);
  if (row >= n) return;
  const float *x = X + row * width;
  const int nblocks = (width + KC - 1) / KC;
  float acc = 0.f;
  for (int b0 = 0; b0 < nblocks; b0 += 32) {
    const int k0 = (b0 + lane) * KC, k1 = min(k0 + KC, width);
    float part = 0.f;
    for (int k = k0; k < k1; ++k) part = fadd(part, fmul(x[k], x[k]));
    const int nb = min(32, nblocks - b0);
    for (int b = 0; b < nb; ++b) acc = fadd(acc, __shfl_sync(0xffffffffu, part, b));
  }
  if (lane == 0) out[row] = fsqrt(acc);
}

// The rows of `table`: pointer, count and width.
static int sim_table(const kge_model_t *m, int table, const float *&X, int64_t &rows, int &width) {
  const int rc = check_model(m);
  if (rc) return rc;
  KGE_REQUIRE(table == KGE_TABLE_ENTITY || table == KGE_TABLE_RELATION,
              "table %d is neither KGE_TABLE_ENTITY nor KGE_TABLE_RELATION", table);
  const bool ent = table == KGE_TABLE_ENTITY;
  X = ent ? m->entity : m->relation;
  rows = ent ? m->nentity : m->nrelation;
  width = (int)(ent ? m->entity_dim : m->relation_dim);
  return KGE_OK;
}

static int sim_check(const kge_model_t *m, int table, int64_t Q, int64_t row_begin, int64_t row_end, int k,
                     const float *&X, int64_t &rows, int &width) {
  const int rc = sim_table(m, table, X, rows, width);
  if (rc) return rc;
  KGE_REQUIRE(k >= 1 && k <= KGE_TOPK_MAX, "k = %d outside [1, %d]", k, KGE_TOPK_MAX);
  KGE_REQUIRE(Q >= 0 && (Q + TQ - 1) / TQ <= 65535, "at most %d queries per call", 65535 * TQ);
  KGE_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= rows, "row slice [%lld,%lld) outside [0,%lld)",
              (long long)row_begin, (long long)row_end, (long long)rows);
  return KGE_OK;
}

static size_t sim_lists_bytes(int64_t Q, int64_t row_begin, int64_t row_end, int k) {
  if (Q == 0 || row_begin == row_end) return 0;
  return sizeof(uint64_t) * (size_t)Q * topk_strips(false, Q, row_end - row_begin, k) * k;
}

}  // namespace kge

using namespace kge;

extern "C" int64_t kge_eval_topk_scratch_bytes(const kge_model_t *m, int64_t Q, int64_t ent_begin, int64_t ent_end,
                                               int k) {
  const int rc = topk_check(m, Q, ent_begin, ent_end, k);
  if (rc) return rc;
  return (int64_t)topk_lists_bytes(m, Q, ent_begin, ent_end, k);
}

extern "C" int kge_eval_topk(const kge_model_t *m, int mode, const float *qvec, int64_t Q, const float *phase_table,
                             const uint32_t *exclude_bits, int64_t ent_begin, int64_t ent_end, int k, uint64_t *keys_out,
                             void *scratch, int64_t scratch_bytes, void *stream) {
  int rc = topk_check(m, Q, ent_begin, ent_end, k);
  if (rc) return rc;
  bool head;
  if ((rc = eval_mode(mode, head))) return rc;
  KGE_REQUIRE(qvec && keys_out, "null pointer");
  const size_t need = topk_lists_bytes(m, Q, ent_begin, ent_end, k);
  KGE_REQUIRE(scratch_bytes >= (int64_t)need && (scratch || need == 0), "scratch of %lld bytes, need %lld",
              (long long)scratch_bytes, (long long)need);
  if (Q == 0) return KGE_OK;
  EvalArgs a{};
  if ((rc = fill_eval_args(m, head, qvec, nullptr, Q, phase_table, a))) return rc;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (ent_begin == ent_end) {                              // nothing to select from: every slot empty
    KGE_CUDA_OK(cudaMemsetAsync(keys_out, 0, sizeof(uint64_t) * (size_t)Q * k, st));
    return KGE_OK;
  }
  a.ent_begin = ent_begin;
  a.ent_end = ent_end;
  const bool cplx = m->model == KGE_COMPLEX || m->model == KGE_ROTATE;
  TopkArgs t{};
  t.exclude = exclude_bits;
  t.lists = (uint64_t *)scratch;
  t.k = k;
  t.strips = topk_strips(cplx, Q, ent_end - ent_begin, k);
  const int64_t ntiles = (ent_end - ent_begin + TJ - 1) / TJ;
  t.tiles_per_strip = (int)((ntiles + t.strips - 1) / t.strips);
  const bool aligned = eval_aligned(a);
#define KGE_TK(OP)                                     \
  case OP:                                             \
    rc = launch_topk<OP, SIM_LINK>(a, t, aligned, st); \
    break;
  switch (op_of(m->model, head)) {
    KGE_TK(OP_SUBABS) KGE_TK(OP_ADDABS) KGE_TK(OP_MUL) KGE_TK(OP_CMUL) KGE_TK(OP_CDIST) KGE_TK(OP_SUBSIN)
    KGE_TK(OP_ADDSIN)
  }
#undef KGE_TK
  if (rc) return rc;
  return launch_merge(t.lists, Q, t.strips, k, keys_out, nullptr, nullptr, st);
}

extern "C" int kge_eval_topk_merge(const uint64_t *keys_in, int64_t Q, int lists, int k, uint64_t *keys_out,
                                   int64_t *ids_out, float *scores_out, void *stream) {
  KGE_REQUIRE(k >= 1 && k <= KGE_TOPK_MAX, "k = %d outside [1, %d]", k, KGE_TOPK_MAX);
  KGE_REQUIRE(lists >= 1 && Q >= 0, "bad sizes");
  KGE_REQUIRE((keys_in || Q == 0) && (keys_out || ids_out || scores_out), "null pointer");
  KGE_REQUIRE(keys_out != keys_in || Q == 0, "keys_out must not alias keys_in");
  if (Q == 0) return KGE_OK;
  return launch_merge(keys_in, Q, lists, k, keys_out, ids_out, scores_out, (cudaStream_t)stream);
}

extern "C" int kge_similarity_rows(const kge_model_t *m, int table, const int64_t *ids, int64_t Q, float *rows_out,
                                   int32_t *err_flag, void *stream) {
  const float *X;
  int64_t rows;
  int width;
  int rc = sim_table(m, table, X, rows, width);
  if (rc) return rc;
  KGE_REQUIRE(Q >= 0, "Q = %lld", (long long)Q);
  KGE_REQUIRE((ids && rows_out) || Q == 0, "null pointer");
  if (Q == 0) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  const int64_t blocks = (Q * width + SIM_THREADS - 1) / SIM_THREADS;
  gather_rows_kernel<<<(unsigned)(blocks < 148 * 32 ? blocks : 148 * 32), SIM_THREADS, 0, (cudaStream_t)stream>>>(
      X, rows, width, ids, Q, rows_out, err_flag);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

extern "C" int kge_similarity_norms(const kge_model_t *m, int table, const float *vectors, int64_t n, float *norms_out,
                                    void *stream) {
  const float *X;
  int64_t rows;
  int width;
  int rc = sim_table(m, table, X, rows, width);
  if (rc) return rc;
  KGE_REQUIRE(vectors || n == rows, "the norms of the table need n = %lld rows, got %lld", (long long)rows, (long long)n);
  KGE_REQUIRE(n >= 0, "n = %lld", (long long)n);
  KGE_REQUIRE(norms_out || n == 0, "null pointer");
  if (n == 0) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  const int64_t blocks = (n + SIM_THREADS / 32 - 1) / (SIM_THREADS / 32);
  row_norms_kernel<<<(unsigned)blocks, SIM_THREADS, 0, (cudaStream_t)stream>>>(vectors ? vectors : X, n, width, norms_out);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

extern "C" int64_t kge_similarity_topk_scratch_bytes(const kge_model_t *m, int table, int64_t Q, int64_t row_begin,
                                                     int64_t row_end, int k) {
  const float *X;
  int64_t rows;
  int width;
  const int rc = sim_check(m, table, Q, row_begin, row_end, k, X, rows, width);
  if (rc) return rc;
  return (int64_t)sim_lists_bytes(Q, row_begin, row_end, k);
}

extern "C" int kge_similarity_topk(const kge_model_t *m, int table, int metric, const float *qvec, const float *qnorm,
                                   const float *xnorm, const int64_t *self_ids, int64_t Q, int64_t row_begin,
                                   int64_t row_end, int k, uint64_t *keys_out, void *scratch, int64_t scratch_bytes,
                                   void *stream) {
  const float *X;
  int64_t rows;
  int width;
  int rc = sim_check(m, table, Q, row_begin, row_end, k, X, rows, width);
  if (rc) return rc;
  KGE_REQUIRE(metric >= KGE_SIM_DOT && metric <= KGE_SIM_L1, "metric %d is not one of KGE_SIM_DOT ... KGE_SIM_L1",
              metric);
  KGE_REQUIRE(qvec && keys_out, "null pointer");
  KGE_REQUIRE(metric != KGE_SIM_COSINE || (qnorm && xnorm), "cosine needs the norms qnorm and xnorm");
  const size_t need = sim_lists_bytes(Q, row_begin, row_end, k);
  KGE_REQUIRE(scratch_bytes >= (int64_t)need && (scratch || need == 0), "scratch of %lld bytes, need %lld",
              (long long)scratch_bytes, (long long)need);
  if (Q == 0) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (row_begin == row_end) {                              // nothing to select from: every slot empty
    KGE_CUDA_OK(cudaMemsetAsync(keys_out, 0, sizeof(uint64_t) * (size_t)Q * k, st));
    return KGE_OK;
  }
  EvalArgs a{};                                            // the real-row path: H = 1, d = De = width
  a.qvec = qvec;
  a.X = X;
  a.Q = Q;
  a.nentity = rows;
  a.ent_begin = row_begin;
  a.ent_end = row_end;
  a.d = a.De = width;
  TopkArgs t{};
  t.lists = (uint64_t *)scratch;
  t.k = k;
  t.strips = topk_strips(false, Q, row_end - row_begin, k);
  const int64_t ntiles = (row_end - row_begin + TJ - 1) / TJ;
  t.tiles_per_strip = (int)((ntiles + t.strips - 1) / t.strips);
  t.qnorm = qnorm;
  t.xnorm = xnorm;
  t.self_ids = self_ids;
  const bool aligned = eval_aligned(a);
  switch (metric) {
    case KGE_SIM_DOT: rc = launch_topk<OP_MUL, KGE_SIM_DOT>(a, t, aligned, st); break;
    case KGE_SIM_COSINE: rc = launch_topk<OP_MUL, KGE_SIM_COSINE>(a, t, aligned, st); break;
    case KGE_SIM_L2: rc = launch_topk<OP_SQDIFF, KGE_SIM_L2>(a, t, aligned, st); break;
    default: rc = launch_topk<OP_SUBABS, KGE_SIM_L1>(a, t, aligned, st); break;
  }
  if (rc) return rc;
  return launch_merge(t.lists, Q, t.strips, k, keys_out, nullptr, nullptr, st);
}
