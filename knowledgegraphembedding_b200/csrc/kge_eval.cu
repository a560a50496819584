// kge_eval.cu -- filtered all-entity ranking without a sort (KGEModel.test_step, model.py:346-427).
//
// The reference scores every entity as a candidate, adds filter_bias, argsorts each row and looks up the
// position of the positive.  The position only depends on how many unfiltered candidates beat the
// positive, so this file computes exactly that count:
//   query_vectors    fold the fixed side of every query into q[Q, D_e]           (model.py:214-223 ...)
//   positive_scores  s_pos[q], bit-identical to the tile kernel's value for that column
//   count_ranks      register-tiled [64 queries x 64 entities] CTA tiles streamed over k through a
//                    double-buffered cp.async pipeline; epilogue compares with s_pos, applies the filter
//                    bitmap and accumulates integer counts (bit-exact, order independent)
// All score arithmetic here is written with un-contractable IEEE primitives and accumulated over k in
// index order, so the CPU oracle (oracle/kge_oracle.c) reproduces every score bit-for-bit.
#include "kge_eval_tile.cuh"

namespace kge {

// ---- query vectors ---------------------------------------------------------------------------------------
template <int MODEL, bool HEAD>
__global__ void query_vectors_kernel(const float *__restrict__ E, const float *__restrict__ R,
                                     const int64_t *__restrict__ queries, int64_t Q, int64_t nentity,
                                     int64_t nrelation, int d, int De, int Dr, float scale,
                                     float *__restrict__ qvec, int32_t *err) {
  for (int64_t qi = blockIdx.x; qi < Q; qi += gridDim.x) {
    int64_t fid = queries[qi * 3 + (HEAD ? 2 : 0)], rid = queries[qi * 3 + 1];
    const int64_t pid = queries[qi * 3 + (HEAD ? 0 : 2)];
    if ((uint64_t)pid >= (uint64_t)nentity && threadIdx.x == 0 && err) *err = 1;
    if ((uint64_t)fid >= (uint64_t)nentity || (uint64_t)rid >= (uint64_t)nrelation) {
      if (threadIdx.x == 0 && err) *err = 1;
      fid = 0; rid = 0;
    }
    const float *F = E + fid * De, *Rr = R + rid * Dr;
    float *q = qvec + qi * De;
    for (int k = threadIdx.x; k < d; k += blockDim.x) build_q<MODEL, HEAD>(F, Rr, k, d, scale, q);
  }
}

__global__ void phase_table_kernel(const float *__restrict__ E, int64_t n, float scale, float *__restrict__ P) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    P[i] = fdiv(E[i], scale);
}

// ---- canonical score of one (query vector, candidate row) pair, computed by a whole warp ------------------------
// Lane l sums block l (32 consecutive k, index order, from 0.0f); lane 0 then adds the block sums in index order.
// Bit-identical to the sequential definition, ~32x shorter dependency chain.  Result valid in every lane.
template <int OP>
__device__ __forceinline__ float canonical_pair_score(const float *__restrict__ q, const float *__restrict__ x, int d) {
  constexpr bool CPLX = op_is_complex(OP);
  const int lane = threadIdx.x & 31;
  const int nblocks = (d + KC - 1) / KC;
  const bool vec4 = (d % 4 == 0) && ((((uintptr_t)q | (uintptr_t)x) & 15) == 0);
  float acc = 0.f;
  for (int b0 = 0; b0 < nblocks; b0 += 32) {
    const int blk = b0 + lane;
    float part = 0.f;
    if (blk < nblocks) {
      const int k0 = blk * KC, k1 = k0 + KC < d ? k0 + KC : d;
      if (vec4) {                                          // 16-byte loads; same element order
        for (int k = k0; k < k1; k += 4) {
          const float4 qa = *reinterpret_cast<const float4 *>(q + k), xa = *reinterpret_cast<const float4 *>(x + k);
          float4 qb = make_float4(0.f, 0.f, 0.f, 0.f), xb = qb;
          if constexpr (CPLX) {
            qb = *reinterpret_cast<const float4 *>(q + d + k);
            xb = *reinterpret_cast<const float4 *>(x + d + k);
          }
          part = fadd(part, op_exact<OP>(qa.x, qb.x, xa.x, xb.x));
          part = fadd(part, op_exact<OP>(qa.y, qb.y, xa.y, xb.y));
          part = fadd(part, op_exact<OP>(qa.z, qb.z, xa.z, xb.z));
          part = fadd(part, op_exact<OP>(qa.w, qb.w, xa.w, xb.w));
        }
      } else {
        for (int k = k0; k < k1; ++k)
          part = fadd(part, op_exact<OP>(q[k], CPLX ? q[d + k] : 0.f, x[k], CPLX ? x[d + k] : 0.f));
      }
    }
    const int nb = nblocks - b0 < 32 ? nblocks - b0 : 32;
    for (int l = 0; l < nb; ++l) acc = fadd(acc, __shfl_sync(0xffffffffu, part, l));
  }
  return acc;
}

// ---- positive scores ----------------------------------------------------------------------------------------
template <int OP>
__global__ void positive_scores_kernel(const float *__restrict__ qvec, const float *__restrict__ X,
                                       const int64_t *__restrict__ queries, int pos_col, int64_t Q, int64_t nentity,
                                       int d, int De, float gamma, const float *__restrict__ modulus,
                                       float *__restrict__ pos_score) {
  const int64_t qi = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;      // one warp per query
  if (qi >= Q) return;
  int64_t pid = queries[qi * 3 + pos_col];
  if ((uint64_t)pid >= (uint64_t)nentity) pid = 0;
  const float acc = canonical_pair_score<OP>(qvec + qi * De, X + pid * De, d);
  if ((threadIdx.x & 31) == 0) pos_score[qi] = finish_exact<OP>(acc, gamma, modulus ? modulus[0] : 1.f);
}

// ---- tiled score + count ---------------------------------------------------------------------------------------
// STATS: a.counts is the [Q, KGE_RANK_STATS] table of kge_eval_count_rank_stats instead of [Q] counts.
template <int OP, bool ALIGNED, bool FAST = false, bool STATS = false>
__global__ void __launch_bounds__(EVAL_THREADS, 2) count_ranks_kernel(const EvalArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ int cnt_sh[STATS ? KGE_RANK_STATS * TQ : TQ];

  const int tid = threadIdx.x;
  const int tq = tid % 16, tj = tid / 16;
  const int64_t j0 = a.ent_begin + (int64_t)blockIdx.x * TJ;
  const int64_t q0 = (int64_t)blockIdx.y * TQ;
  if constexpr (STATS) {
    for (int i = tid; i < KGE_RANK_STATS * TQ; i += EVAL_THREADS) cnt_sh[i] = 0;
  } else {
    if (tid < TQ) cnt_sh[tid] = 0;
  }

  const TileAcc t = tile_mainloop<OP, ALIGNED, FAST>(a, smem, q0, j0, tq, tj);
  const auto &acc = t.v;

  const float modulus = a.modulus ? a.modulus[0] : 1.f;
  [[maybe_unused]] const FastBand band = fast_band(OP != OP_CDIST, a.d, modulus);
  if constexpr (STATS) {
    // ---- epilogue: the six counters of every column but the positive's; a filtered column keeps its own score ----
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t qi = q0 + tq + 16 * i;
      if (qi >= a.Q) continue;
      const float sp = a.pos_score[qi];
      const int64_t pid = a.queries[qi * 3 + a.pos_col];
      int c[KGE_RANK_STATS] = {0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t ej = j0 + tj + 16 * j;
        if (ej >= a.ent_end || ej == pid) continue;
        const float s = finish_exact<OP>(acc[i][j], a.gamma, modulus);
        const bool kept = !((a.filter_bits[qi * a.words + (ej >> 5)] >> (ej & 31)) & 1u);
        if constexpr (FAST) {                            // s is only within eps of the canonical score
          const float eps = fast_eps(band, a.gamma, s);
          if (s - eps > sp) {
            c[0] += kept;
            ++c[3];
          } else if (!(s + eps < sp)) {                  // equal, undecidable here, or NaN: exact re-score later
            const int slot = atomicAdd(a.amb_count, 1);
            if (slot < a.amb_capacity) a.amb[slot] = make_int2((int)qi, (int)ej);
            else a.amb_count[1] = 1;
          }
        } else {
          const bool gt = s > sp, eb = s == sp && ej < pid, ea = s == sp && ej > pid;
          c[0] += kept && gt;
          c[1] += kept && eb;
          c[2] += kept && ea;
          c[3] += gt;
          c[4] += eb;
          c[5] += ea;
        }
      }
#pragma unroll
      for (int k = 0; k < KGE_RANK_STATS; ++k)
        if (c[k]) atomicAdd(&cnt_sh[(tq + 16 * i) * KGE_RANK_STATS + k], c[k]);
    }
    __syncthreads();
    for (int i = tid; i < KGE_RANK_STATS * TQ; i += EVAL_THREADS)
      if (cnt_sh[i] && q0 + i / KGE_RANK_STATS < a.Q) atomicAdd(&a.counts[q0 * KGE_RANK_STATS + i], cnt_sh[i]);
  } else {
    // ---- epilogue: compare with the positive, apply the filter, count -------------------------------------------
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t qi = q0 + tq + 16 * i;
      if (qi >= a.Q) continue;
      const float sp = a.pos_score[qi];
      int64_t pid = a.queries[qi * 3 + a.pos_col];
      int c = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t ej = j0 + tj + 16 * j;
        if (ej >= a.ent_end) continue;
        float s = finish_exact<OP>(acc[i][j], a.gamma, modulus);
        const bool filtered = ej != pid && ((a.filter_bits[qi * a.words + (ej >> 5)] >> (ej & 31)) & 1u);
        if (filtered) s = fadd(sp, -1.0f);                   // candidate replaced by the positive, bias -1
        else if (ej != pid) {
          if constexpr (FAST) {                              // s is only within eps of the canonical score
            const float eps = fast_eps(band, a.gamma, s);
            if (s - eps > sp) ++c;
            else if (!(s + eps < sp)) {                      // undecidable here (or NaN): exact re-score later
              const int slot = atomicAdd(a.amb_count, 1);
              if (slot < a.amb_capacity) a.amb[slot] = make_int2((int)qi, (int)ej);
              else a.amb_count[1] = 1;
            }
          } else {
            c += (s > sp) || (s == sp && ej < pid);
          }
        }
        if (a.scores_out) a.scores_out[qi * a.nentity + ej] = s;
      }
      if (c) atomicAdd(&cnt_sh[tq + 16 * i], c);
    }
    __syncthreads();
    if (tid < TQ && cnt_sh[tid] && q0 + tid < a.Q) atomicAdd(&a.counts[q0 + tid], cnt_sh[tid]);
  }
}

// exact canonical re-score of a list of ambiguous (query, entity) pairs (tcgen05 path, kge_eval_gemm.cu)
template <int OP>
__global__ void rescore_pairs_kernel(const int2 *__restrict__ amb, const int *__restrict__ amb_count, int capacity,
                                     const float *__restrict__ qvec, const float *__restrict__ E, int d, int De,
                                     const float *__restrict__ pos_score, const int64_t *__restrict__ queries,
                                     int pos_col, float gamma, int32_t *__restrict__ counts,
                                     const float *__restrict__ modulus = nullptr) {
  int n = amb_count[0];
  if (n > capacity) n = capacity;
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  for (int i = wid; i < n; i += nw) {
    const int2 p = amb[i];
    const float s = finish_exact<OP>(canonical_pair_score<OP>(qvec + (int64_t)p.x * De, E + (int64_t)p.y * De, d),
                                     gamma, modulus ? modulus[0] : 1.f);
    if (lane == 0) {
      const float sp = pos_score[p.x];
      const int64_t pid = queries[(int64_t)p.x * 3 + pos_col];
      if (s > sp || (s == sp && p.y < pid)) atomicAdd(counts + p.x, 1);
    }
  }
}

// The same for the stats kernels: each pair (never the positive's column) is classified by the filter bitmap and
// settled as greater / equal before / equal after the positive; stats is [Q, KGE_RANK_STATS].
template <int OP>
__global__ void rescore_pair_stats_kernel(const int2 *__restrict__ amb, const int *__restrict__ amb_count, int capacity,
                                          const float *__restrict__ qvec, const float *__restrict__ E, int d, int De,
                                          const float *__restrict__ pos_score, const int64_t *__restrict__ queries,
                                          int pos_col, float gamma, const float *__restrict__ modulus,
                                          const uint32_t *__restrict__ filter_bits, int words,
                                          int32_t *__restrict__ stats) {
  int n = amb_count[0];
  if (n > capacity) n = capacity;
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  for (int i = wid; i < n; i += nw) {
    const int2 p = amb[i];
    const float s = finish_exact<OP>(canonical_pair_score<OP>(qvec + (int64_t)p.x * De, E + (int64_t)p.y * De, d),
                                     gamma, modulus ? modulus[0] : 1.f);
    if (lane == 0) {
      const float sp = pos_score[p.x];
      const int64_t pid = queries[(int64_t)p.x * 3 + pos_col];
      const int k = s > sp ? 0 : s == sp ? (p.y < pid ? 1 : 2) : -1;
      if (k >= 0) {
        int32_t *row = stats + (int64_t)p.x * KGE_RANK_STATS;
        if (!((filter_bits[(int64_t)p.x * words + (p.y >> 5)] >> (p.y & 31)) & 1u)) atomicAdd(row + k, 1);
        atomicAdd(row + k + 3, 1);
      }
    }
  }
}

// filter_bits non-null: the stats re-score (counts is then [Q, KGE_RANK_STATS])
int launch_rescore_pairs(bool cplx, const void *amb, const int *amb_count, int capacity, const float *qvec,
                         const float *E, int d, int De, const float *pos_score, const int64_t *queries, int pos_col,
                         int32_t *counts, cudaStream_t st, const uint32_t *filter_bits, int words) {
  if (filter_bits) {
    if (cplx)
      rescore_pair_stats_kernel<OP_CMUL><<<148 * 8, 256, 0, st>>>((const int2 *)amb, amb_count, capacity, qvec, E, d, De,
                                                                  pos_score, queries, pos_col, 0.f, nullptr,
                                                                  filter_bits, words, counts);
    else
      rescore_pair_stats_kernel<OP_MUL><<<148 * 8, 256, 0, st>>>((const int2 *)amb, amb_count, capacity, qvec, E, d, De,
                                                                 pos_score, queries, pos_col, 0.f, nullptr,
                                                                 filter_bits, words, counts);
  } else if (cplx)
    rescore_pairs_kernel<OP_CMUL><<<148 * 8, 256, 0, st>>>((const int2 *)amb, amb_count, capacity, qvec, E, d, De,
                                                           pos_score, queries, pos_col, 0.f, counts);
  else
    rescore_pairs_kernel<OP_MUL><<<148 * 8, 256, 0, st>>>((const int2 *)amb, amb_count, capacity, qvec, E, d, De,
                                                          pos_score, queries, pos_col, 0.f, counts);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

__global__ void filter_bits_kernel(const int64_t *__restrict__ offsets, const int32_t *__restrict__ ents, int64_t Q,
                                   int64_t nentity, int words, uint32_t *__restrict__ bits) {
  for (int64_t qi = blockIdx.x; qi < Q; qi += gridDim.x) {
    const int64_t b = offsets[qi], e = offsets[qi + 1];
    for (int64_t i = b + threadIdx.x; i < e; i += blockDim.x) {
      const int32_t j = ents[i];
      if (j >= 0 && j < nentity) atomicOr(&bits[qi * words + (j >> 5)], 1u << (j & 31));
    }
  }
}

// Filter bitmap straight from the device-resident index of all true triples: one CTA per query looks its key
// ((r, t) for head-batch, (h, r) for tail-batch) up in the sorted key table and sets the bits of that key's run.
__global__ void filter_lookup_kernel(const int64_t *__restrict__ keys, const int64_t *__restrict__ key_offsets,
                                     const int32_t *__restrict__ values, int64_t nkeys,
                                     const int64_t *__restrict__ queries, int64_t Q, int head_batch, int64_t nentity,
                                     int64_t nrelation, int words, uint32_t *__restrict__ bits) {
  __shared__ int64_t run[2];
  for (int64_t qi = blockIdx.x; qi < Q; qi += gridDim.x) {
    if (threadIdx.x == 0) {
      const int64_t h = queries[qi * 3], r = queries[qi * 3 + 1], t = queries[qi * 3 + 2];
      const int64_t key = head_batch ? r * nentity + t : h * nrelation + r;
      int64_t lo = 0, hi = nkeys;                                      // lower bound
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (keys[mid] < key) lo = mid + 1; else hi = mid;
      }
      const bool found = lo < nkeys && keys[lo] == key;
      run[0] = found ? key_offsets[lo] : 0;
      run[1] = found ? key_offsets[lo + 1] : 0;
    }
    __syncthreads();
    const int64_t b = run[0], e = run[1];
    for (int64_t i = b + threadIdx.x; i < e; i += blockDim.x) {
      const int32_t j = values[i];
      if (j >= 0 && j < nentity) atomicOr(&bits[qi * words + (j >> 5)], 1u << (j & 31));
    }
    __syncthreads();
  }
}

// ---- device-side build of the filter index (dataloader.py:122-162 keeps all true triples in a python set and probes it
// once per entity per query): a direct-address CSR over the key space nentity x nrelation, by counting sort --
// histogram of the keys, tiled exclusive scan (the train path's scan kernels), scatter.  offsets[key] .. offsets[key + 1]
// then delimit the true heads of (r, t) / true tails of (h, r); no sorted key table, no binary search per query.
__global__ void __launch_bounds__(1024) scan_tiles_kernel(const int *__restrict__ cnt, int *__restrict__ cursor,
                                                          int *__restrict__ tile_tot, int64_t n);      // kge_train.cu
__global__ void __launch_bounds__(1024) scan_apply_kernel(int *__restrict__ cnt, int *__restrict__ cursor,
                                                          const int *__restrict__ tile_tot, int64_t n);

template <bool PLACE>
__global__ void filter_index_kernel(const int64_t *__restrict__ tri, int64_t n, int head_batch, int64_t nentity,
                                    int64_t nrelation, int *__restrict__ cnt_or_cursor, int32_t *__restrict__ entities,
                                    int32_t *err) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t h = tri[3 * i], r = tri[3 * i + 1], t = tri[3 * i + 2];
    if ((uint64_t)h >= (uint64_t)nentity || (uint64_t)t >= (uint64_t)nentity || (uint64_t)r >= (uint64_t)nrelation) {
      if (err) *err = 1;                                   // (a triple outside the tables can never be a query's answer)
      continue;
    }
    const int64_t key = head_batch ? r * nentity + t : h * nrelation + r;
    const int pos = atomicAdd(cnt_or_cursor + key, 1);
    if (PLACE) entities[pos] = (int32_t)(head_batch ? h : t);
  }
}

__global__ void filter_lookup_dense_kernel(const int32_t *__restrict__ offsets, const int32_t *__restrict__ values,
                                           const int64_t *__restrict__ queries, int64_t Q, int head_batch,
                                           int64_t nentity, int64_t nrelation, int words, uint32_t *__restrict__ bits) {
  for (int64_t qi = blockIdx.x; qi < Q; qi += gridDim.x) {
    const int64_t h = queries[qi * 3], r = queries[qi * 3 + 1], t = queries[qi * 3 + 2];
    const int64_t fixed = head_batch ? t : h;
    if ((uint64_t)fixed >= (uint64_t)nentity || (uint64_t)r >= (uint64_t)nrelation) continue;   // flagged by the query kernels
    const int64_t key = head_batch ? r * nentity + t : h * nrelation + r;
    const int b = offsets[key], e = offsets[key + 1];
    for (int i = b + threadIdx.x; i < e; i += blockDim.x) {
      const int32_t j = values[i];
      atomicOr(&bits[qi * words + (j >> 5)], 1u << (j & 31));
    }
  }
}

template <int OP, bool STATS>
static int launch_count(const EvalArgs &a, bool aligned, cudaStream_t st) {
  constexpr int H = op_is_complex(OP) ? 2 : 1;
  const size_t smem = sizeof(float) * 2 * (TQ + TJ) * H * ST;
  dim3 grid((unsigned)((a.ent_end - a.ent_begin + TJ - 1) / TJ), (unsigned)((a.Q + TQ - 1) / TQ));
  if constexpr (OP == OP_CDIST || OP == OP_SUBSIN || OP == OP_ADDSIN) {
    if (a.amb && aligned && a.d <= kFastMaxD) {                      // two-stage: fast tile pass + exact re-score
      KGE_CUDA_OK(cudaMemsetAsync(a.amb_count, 0, 2 * sizeof(int), st));
      auto k = count_ranks_kernel<OP, true, true, STATS>;
      KGE_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k<<<grid, EVAL_THREADS, smem, st>>>(a);
      KGE_CUDA_OK(cudaGetLastError());
      if constexpr (STATS)
        rescore_pair_stats_kernel<OP><<<148 * 4, 256, 0, st>>>(a.amb, a.amb_count, a.amb_capacity, a.qvec, a.X, a.d,
                                                               a.De, a.pos_score, a.queries, a.pos_col, a.gamma,
                                                               a.modulus, a.filter_bits, a.words, a.counts);
      else
        rescore_pairs_kernel<OP><<<148 * 4, 256, 0, st>>>(a.amb, a.amb_count, a.amb_capacity, a.qvec, a.X, a.d, a.De,
                                                          a.pos_score, a.queries, a.pos_col, a.gamma, a.counts, a.modulus);
      KGE_CUDA_OK(cudaGetLastError());
      return KGE_OK;
    }
  }
  if (aligned) {
    auto k = count_ranks_kernel<OP, true, false, STATS>;
    KGE_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, EVAL_THREADS, smem, st>>>(a);
  } else {
    auto k = count_ranks_kernel<OP, false, false, STATS>;
    KGE_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, EVAL_THREADS, smem, st>>>(a);
  }
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

}  // namespace kge

using namespace kge;

extern "C" int kge_eval_query_vectors(const kge_model_t *m, int mode, const int64_t *queries, int64_t Q, float *qvec,
                                      int32_t *err_flag, void *stream) {
  int rc = check_model(m);
  if (rc) return rc;
  bool head;
  if ((rc = eval_mode(mode, head))) return rc;
  KGE_REQUIRE(queries && qvec, "null pointer");
  if (Q <= 0) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  const bool cplx = m->model == KGE_COMPLEX || m->model == KGE_ROTATE;
  const int d = cplx ? (int)(m->entity_dim / 2) : (int)m->entity_dim;
  const int grid = (int)(Q < 148 * 16 ? Q : 148 * 16);
  const float scale = phase_scale(m);
  cudaStream_t st = (cudaStream_t)stream;
#define KGE_QV(MODEL)                                                                                              \
  case MODEL:                                                                                                      \
    if (head)                                                                                                      \
      query_vectors_kernel<MODEL, true><<<grid, 256, 0, st>>>(m->entity, m->relation, queries, Q, m->nentity,       \
                                                              m->nrelation, d, (int)m->entity_dim,                 \
                                                              (int)m->relation_dim, scale, qvec, err_flag);        \
    else                                                                                                           \
      query_vectors_kernel<MODEL, false><<<grid, 256, 0, st>>>(m->entity, m->relation, queries, Q, m->nentity,      \
                                                               m->nrelation, d, (int)m->entity_dim,                \
                                                               (int)m->relation_dim, scale, qvec, err_flag);       \
    break;
  switch (m->model) {
    KGE_QV(KGE_TRANSE)
    KGE_QV(KGE_DISTMULT)
    KGE_QV(KGE_COMPLEX)
    KGE_QV(KGE_ROTATE)
    KGE_QV(KGE_PROTATE)
  }
#undef KGE_QV
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

extern "C" int kge_eval_phase_table(const kge_model_t *m, float *phase_table, void *stream) {
  int rc = check_model(m);
  if (rc) return rc;
  KGE_REQUIRE(phase_table, "null pointer");
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  phase_table_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(m->entity, m->nentity * m->entity_dim, phase_scale(m),
                                                              phase_table);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

extern "C" int kge_eval_positive_scores(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                                        int64_t Q, const float *phase_table, float *pos_score, void *stream) {
  int rc = check_model(m);
  if (rc) return rc;
  bool head;
  if ((rc = eval_mode(mode, head))) return rc;
  KGE_REQUIRE(qvec && queries && pos_score, "null pointer");
  if (Q <= 0) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  EvalArgs a{};
  if ((rc = fill_eval_args(m, head, qvec, queries, Q, phase_table, a))) return rc;
  const int grid = (int)((Q + 3) / 4);                   // 4 warps per CTA, one warp per query
  cudaStream_t st = (cudaStream_t)stream;
#define KGE_PS(OP)                                                                                              \
  case OP:                                                                                                      \
    positive_scores_kernel<OP><<<grid, 128, 0, st>>>(a.qvec, a.X, a.queries, a.pos_col, a.Q, a.nentity, a.d, a.De, \
                                                     a.gamma, a.modulus, pos_score);                            \
    break;
  switch (op_of(m->model, head)) {
    KGE_PS(OP_SUBABS) KGE_PS(OP_ADDABS) KGE_PS(OP_MUL) KGE_PS(OP_CMUL) KGE_PS(OP_CDIST) KGE_PS(OP_SUBSIN)
    KGE_PS(OP_ADDSIN)
  }
#undef KGE_PS
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

static int count_ranks_impl(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries, int64_t Q,
                            const float *phase_table, const float *pos_score, const uint32_t *filter_bits,
                            int64_t ent_begin, int64_t ent_end, int32_t *counts, float *scores_out, void *amb_pairs,
                            int64_t amb_capacity, int32_t *amb_count, void *stream, bool stats = false);

extern "C" int kge_eval_count_ranks(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries, int64_t Q,
                                    const float *phase_table, const float *pos_score, const uint32_t *filter_bits,
                                    int64_t ent_begin, int64_t ent_end, int32_t *counts, float *scores_out,
                                    void *stream) {
  return count_ranks_impl(m, mode, qvec, queries, Q, phase_table, pos_score, filter_bits, ent_begin, ent_end, counts,
                          scores_out, nullptr, 0, nullptr, stream);
}

extern "C" int kge_eval_count_ranks_two_stage(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                                              int64_t Q, const float *phase_table, const float *pos_score,
                                              const uint32_t *filter_bits, int64_t ent_begin, int64_t ent_end,
                                              int32_t *counts, void *amb_pairs, int64_t amb_capacity,
                                              int32_t *amb_count, void *stream) {
  return kge_eval_count_ranks_two_stage_approx(m, mode, qvec, queries, Q, phase_table, pos_score, filter_bits, ent_begin,
                                               ent_end, counts, amb_pairs, amb_capacity, amb_count, nullptr, stream);
}

extern "C" int kge_eval_count_ranks_two_stage_approx(const kge_model_t *m, int mode, const float *qvec,
                                                     const int64_t *queries, int64_t Q, const float *phase_table,
                                                     const float *pos_score, const uint32_t *filter_bits,
                                                     int64_t ent_begin, int64_t ent_end, int32_t *counts,
                                                     void *amb_pairs, int64_t amb_capacity, int32_t *amb_count,
                                                     float *approx_scores_out, void *stream) {
  KGE_REQUIRE(amb_pairs && amb_count && amb_capacity > 0, "two-stage ranking needs the ambiguous-pair buffers");
  // the fast pass writes its own scores through scores_out (only this entry sets both scores_out and the pair list)
  return count_ranks_impl(m, mode, qvec, queries, Q, phase_table, pos_score, filter_bits, ent_begin, ent_end, counts,
                          approx_scores_out, amb_pairs, amb_capacity, amb_count, stream);
}

extern "C" int kge_eval_count_rank_stats(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                                         int64_t Q, const float *phase_table, const float *pos_score,
                                         const uint32_t *filter_bits, int64_t ent_begin, int64_t ent_end, int32_t *stats,
                                         void *stream) {
  return count_ranks_impl(m, mode, qvec, queries, Q, phase_table, pos_score, filter_bits, ent_begin, ent_end, stats,
                          nullptr, nullptr, 0, nullptr, stream, true);
}

extern "C" int kge_eval_count_rank_stats_two_stage(const kge_model_t *m, int mode, const float *qvec,
                                                   const int64_t *queries, int64_t Q, const float *phase_table,
                                                   const float *pos_score, const uint32_t *filter_bits,
                                                   int64_t ent_begin, int64_t ent_end, int32_t *stats, void *amb_pairs,
                                                   int64_t amb_capacity, int32_t *amb_count, void *stream) {
  KGE_REQUIRE(amb_pairs && amb_count && amb_capacity > 0, "two-stage ranking needs the ambiguous-pair buffers");
  return count_ranks_impl(m, mode, qvec, queries, Q, phase_table, pos_score, filter_bits, ent_begin, ent_end, stats,
                          nullptr, amb_pairs, amb_capacity, amb_count, stream, true);
}

extern "C" int kge_eval_two_stage_band(int model, int64_t entity_dim, float modulus, float *host_band) {
  KGE_REQUIRE(host_band, "null pointer");
  KGE_REQUIRE(model == KGE_ROTATE || model == KGE_PROTATE, "model %d has no two-stage pass", model);
  const int64_t d = model == KGE_ROTATE ? entity_dim / 2 : entity_dim;
  KGE_REQUIRE(entity_dim > 0 && (model != KGE_ROTATE || entity_dim % 2 == 0) && d <= kFastMaxD,
              "entity_dim %lld has no two-stage pass (d at most %d)", (long long)entity_dim, kFastMaxD);
  const FastBand b = fast_band(model == KGE_PROTATE, (int)d, modulus);
  host_band[0] = b.c_abs;
  host_band[1] = b.c_rel;
  host_band[2] = b.c_ulp;
  return KGE_OK;
}

static int count_ranks_impl(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries, int64_t Q,
                            const float *phase_table, const float *pos_score, const uint32_t *filter_bits,
                            int64_t ent_begin, int64_t ent_end, int32_t *counts, float *scores_out, void *amb_pairs,
                            int64_t amb_capacity, int32_t *amb_count, void *stream, bool stats) {
  int rc = check_model(m);
  if (rc) return rc;
  bool head;
  if ((rc = eval_mode(mode, head))) return rc;
  KGE_REQUIRE(qvec && queries && pos_score && filter_bits && counts, "null pointer");
  KGE_REQUIRE(ent_begin >= 0 && ent_begin <= ent_end && ent_end <= m->nentity, "entity slice [%lld,%lld) outside [0,%lld)",
              (long long)ent_begin, (long long)ent_end, (long long)m->nentity);
  if (Q <= 0 || ent_begin == ent_end) return KGE_OK;
  KGE_REQUIRE((Q + TQ - 1) / TQ <= 65535, "at most %d queries per call", 65535 * TQ);
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  EvalArgs a{};
  if ((rc = fill_eval_args(m, head, qvec, queries, Q, phase_table, a))) return rc;
  a.pos_score = pos_score; a.filter_bits = filter_bits; a.counts = counts; a.scores_out = scores_out;
  a.ent_begin = ent_begin; a.ent_end = ent_end;
  a.amb = (int2 *)amb_pairs; a.amb_count = amb_count; a.amb_capacity = (int)amb_capacity;
  const bool aligned = eval_aligned(a);
  cudaStream_t st = (cudaStream_t)stream;
#define KGE_CR(OP) \
  case OP:         \
    return stats ? launch_count<OP, true>(a, aligned, st) : launch_count<OP, false>(a, aligned, st);
  switch (op_of(m->model, head)) {
    KGE_CR(OP_SUBABS) KGE_CR(OP_ADDABS) KGE_CR(OP_MUL) KGE_CR(OP_CMUL) KGE_CR(OP_CDIST) KGE_CR(OP_SUBSIN)
    KGE_CR(OP_ADDSIN)
  }
#undef KGE_CR
  set_error("unreachable");
  return KGE_ERR_INVALID;
}

extern "C" int kge_eval_filter_bits(const int64_t *csr_offsets, const int32_t *csr_entities, int64_t Q, int64_t nentity,
                                    uint32_t *filter_bits, void *stream) {
  KGE_REQUIRE(csr_offsets && filter_bits && Q >= 0 && nentity > 0, "bad arguments");
  if (Q == 0) return KGE_OK;
  const int words = (int)((nentity + 31) / 32);
  cudaStream_t st = (cudaStream_t)stream;
  KGE_CUDA_OK(cudaMemsetAsync(filter_bits, 0, sizeof(uint32_t) * (size_t)Q * words, st));
  const int grid = (int)(Q < 148 * 16 ? Q : 148 * 16);
  filter_bits_kernel<<<grid, 128, 0, st>>>(csr_offsets, csr_entities, Q, nentity, words, filter_bits);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

extern "C" int kge_eval_filter_bits_lookup(const int64_t *index_keys, const int64_t *index_offsets,
                                           const int32_t *index_entities, int64_t nkeys, const int64_t *queries,
                                           int64_t Q, int mode, int64_t nentity, int64_t nrelation,
                                           uint32_t *filter_bits, void *stream) {
  KGE_REQUIRE(filter_bits && queries && Q >= 0 && nentity > 0 && nrelation > 0 && nkeys >= 0, "bad arguments");
  KGE_REQUIRE(nkeys == 0 || (index_keys && index_offsets && index_entities), "null filter index");
  KGE_REQUIRE(mode == KGE_HEAD_BATCH || mode == KGE_TAIL_BATCH, "negative batch mode %d not supported", mode);
  if (Q == 0) return KGE_OK;
  const int words = (int)((nentity + 31) / 32);
  cudaStream_t st = (cudaStream_t)stream;
  KGE_CUDA_OK(cudaMemsetAsync(filter_bits, 0, sizeof(uint32_t) * (size_t)Q * words, st));
  if (nkeys == 0) return KGE_OK;
  const int grid = (int)(Q < 148 * 16 ? Q : 148 * 16);
  filter_lookup_kernel<<<grid, 128, 0, st>>>(index_keys, index_offsets, index_entities, nkeys, queries, Q,
                                             mode == KGE_HEAD_BATCH, nentity, nrelation, words, filter_bits);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

static size_t align256e(size_t x) { return (x + 255) & ~(size_t)255; }

extern "C" int64_t kge_eval_filter_index_scratch_bytes(int64_t nentity, int64_t nrelation) {
  if (nentity <= 0 || nrelation <= 0) return 0;
  const int64_t nkeys = nentity * nrelation;
  return (int64_t)(align256e((size_t)nkeys * 4) + align256e((size_t)((nkeys + 1023) / 1024) * 4));
}

extern "C" int kge_eval_filter_index_build(const int64_t *triples, int64_t ntriples, int mode, int64_t nentity,
                                           int64_t nrelation, int32_t *offsets, int32_t *entities, void *scratch,
                                           int64_t scratch_bytes, int32_t *err_flag, void *stream) {
  KGE_REQUIRE(mode == KGE_HEAD_BATCH || mode == KGE_TAIL_BATCH, "negative batch mode %d not supported", mode);
  KGE_REQUIRE(nentity > 0 && nrelation > 0 && ntriples >= 0 && ntriples < (1ll << 31), "bad sizes");
  const int64_t nkeys = nentity * nrelation;
  KGE_REQUIRE(nkeys < (1ll << 31) - 1024, "key space of %lld entries is too large for the direct-address index",
              (long long)nkeys);
  KGE_REQUIRE(offsets && scratch && (entities || ntriples == 0) && (triples || ntriples == 0), "null pointer");
  KGE_REQUIRE(scratch_bytes >= kge_eval_filter_index_scratch_bytes(nentity, nrelation), "scratch too small");
  cudaStream_t st = (cudaStream_t)stream;
  int *cnt = offsets;
  int *cursor = (int *)scratch;
  int *tile_tot = (int *)((char *)scratch + align256e((size_t)nkeys * 4));
  KGE_CUDA_OK(cudaMemsetAsync(cnt, 0, (size_t)(nkeys + 1) * 4, st));
  int grid = (int)((ntriples + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  if (grid < 1) grid = 1;
  const int head = mode == KGE_HEAD_BATCH;
  filter_index_kernel<false><<<grid, 256, 0, st>>>(triples, ntriples, head, nentity, nrelation, cnt, nullptr, err_flag);
  KGE_CUDA_OK(cudaGetLastError());
  const int tiles = (int)((nkeys + 1023) / 1024);
  scan_tiles_kernel<<<tiles, 1024, 0, st>>>(cnt, cursor, tile_tot, nkeys);
  KGE_CUDA_OK(cudaGetLastError());
  scan_apply_kernel<<<tiles, 1024, 0, st>>>(cnt, cursor, tile_tot, nkeys);
  KGE_CUDA_OK(cudaGetLastError());
  filter_index_kernel<true><<<grid, 256, 0, st>>>(triples, ntriples, head, nentity, nrelation, cursor, entities, nullptr);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

extern "C" int kge_eval_filter_bits_lookup_dense(const int32_t *index_offsets, const int32_t *index_entities,
                                                 const int64_t *queries, int64_t Q, int mode, int64_t nentity,
                                                 int64_t nrelation, uint32_t *filter_bits, void *stream) {
  KGE_REQUIRE(mode == KGE_HEAD_BATCH || mode == KGE_TAIL_BATCH, "negative batch mode %d not supported", mode);
  KGE_REQUIRE(index_offsets && index_entities && filter_bits && Q >= 0 && nentity > 0 && nrelation > 0, "bad arguments");
  KGE_REQUIRE(queries || Q == 0, "null pointer");
  if (Q == 0) return KGE_OK;
  const int words = (int)((nentity + 31) / 32);
  cudaStream_t st = (cudaStream_t)stream;
  KGE_CUDA_OK(cudaMemsetAsync(filter_bits, 0, sizeof(uint32_t) * (size_t)Q * words, st));
  const int grid = (int)(Q < 148 * 16 ? Q : 148 * 16);
  filter_lookup_dense_kernel<<<grid, 128, 0, st>>>(index_offsets, index_entities, queries, Q, mode == KGE_HEAD_BATCH,
                                                   nentity, nrelation, words, filter_bits);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}
