// kge_train_kernels.cuh -- the two-sweep row kernels (direct loads and TMA ring); see kge_train.cu for the phases.
#pragma once
#include "kge_train_args.cuh"

namespace kge {

constexpr int kChunks = 8;     // units per lane per k-tile: 8 x float4 x (re,im) = 64 accumulator registers

template <int V>
__device__ __forceinline__ void load_global(float (&o)[V], const float *p) {
  if constexpr (V == 4) {
    float4 t = ldg_stream4(p);
    o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
  } else {
    o[0] = __ldg(p);
  }
}
template <int V>
__device__ __forceinline__ void load_shared(float (&o)[V], const float *p) {
  if constexpr (V == 4) {
    float4 t = *reinterpret_cast<const float4 *>(p);
    o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
  } else {
    o[0] = *p;
  }
}
template <int V>
__device__ __forceinline__ void red_global(float *p, const float (&v)[V]) {
  if constexpr (V == 4) red_add4(p, v[0], v[1], v[2], v[3]);
  else red_add1(p, v[0]);
}

__device__ __forceinline__ float block_reduce(float v, float *scratch, bool is_max) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = is_max ? warp_max(v) : warp_sum(v);
  __syncthreads();                       // protect scratch from the previous use
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  float r = is_max ? -INFINITY : 0.f;
  for (int w = 0; w < nw; ++w) r = is_max ? fmaxf(r, scratch[w]) : r + scratch[w];   // fixed order
  return r;
}

template <int MODEL, bool HEAD, int V>
__global__ void __launch_bounds__(512, 1) row_kernel(const RowArgs a) {
  constexpr int OP = op_of(MODEL, HEAD);
  constexpr bool CPLX = op_is_complex(OP);
  constexpr int H = CPLX ? 2 : 1;              // halves per unit
  extern __shared__ __align__(16) float smem[];
  const int Dq = CPLX ? 2 * a.d : a.d;
  float *q = smem;                             // [Dq]
  float *dq = q + ((Dq + 3) & ~3);             // [Dq]
  float *sc = dq + ((Dq + 3) & ~3);            // [N] scores (only when do_loss)
  float *gg = sc + (a.do_loss ? a.N : 0);      // [N] dL/ds   (only when do_loss)
  float *scratch = gg + (a.do_loss ? a.N : 0); // [32]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int nunits = a.d / V;                  // host guarantees divisibility
  const float modulus = MODEL == KGE_PROTATE ? __ldg(a.modulus) : 1.f;
  const bool do_bwd = a.gE != nullptr;

  for (int rl = blockIdx.x; rl < a.row_count; rl += gridDim.x) {
    const int64_t b = a.row_begin + rl;
    int64_t hid = a.positive[b * 3 + 0], rid = a.positive[b * 3 + 1], tidx = a.positive[b * 3 + 2];
    int64_t fid = HEAD ? tidx : hid;
    if ((uint64_t)fid >= (uint64_t)a.nentity || (uint64_t)rid >= (uint64_t)a.nrelation) {
      if (tid == 0 && a.err) *a.err = 1;
      fid = 0; rid = 0;
    }
    const float *F = a.E + fid * a.De;
    const float *Rr = a.R + rid * a.Dr;
    const int64_t *cand = a.cand + b * a.cand_stride;

    // ---- phase 0: query vector -------------------------------------------------------------------
    __syncthreads();
    for (int k = tid; k < a.d; k += blockDim.x) {
      build_q<MODEL, HEAD>(F, Rr, k, a.d, a.scale, q);
      dq[k] = 0.f;
      if (CPLX) dq[a.d + k] = 0.f;
    }
    __syncthreads();

    // ---- phase 1: scores -------------------------------------------------------------------------
    if (a.do_loss || a.score_out) {
      for (int n = warp; n < a.N; n += nwarps) {
        int64_t id = cand[n];
        if ((uint64_t)id >= (uint64_t)a.nentity) { if (lane == 0 && a.err) *a.err = 1; id = 0; }
        const float *x = a.E + id * a.De;
        float part = 0.f;
        for (int kt = 0; kt < nunits; kt += 32 * kChunks) {
#pragma unroll
          for (int i = 0; i < kChunks; ++i) {
            const int u = kt + lane + 32 * i;
            if (u < nunits) {
              float x0[V], x1[V], q0[V], q1[V];
              load_global<V>(x0, x + u * V);
              load_shared<V>(q0, q + u * V);
              if constexpr (CPLX) {
                load_global<V>(x1, x + a.d + u * V);
                load_shared<V>(q1, q + a.d + u * V);
              }
#pragma unroll
              for (int j = 0; j < V; ++j)
                part += op_forward<OP>(q0[j], CPLX ? q1[j] : 0.f, x0[j], CPLX ? x1[j] : 0.f, a.scale);
            }
          }
        }
        part = warp_sum(part);
        const float s = finish_score<MODEL>(part, a.gamma, modulus);
        if (lane == 0) {
          if (a.do_loss) sc[n] = s;
          if (a.score_out) a.score_out[(int64_t)rl * a.N + n] = s;
        }
      }
    }
    if (!a.do_loss && !do_bwd) continue;

    // ---- phase 2: loss of this row (model.py:270-288) and dL/ds ---------------------------------------
    if (a.do_loss) {
      __syncthreads();
      const float u = a.weight ? a.weight[b] / a.wsum[0] : a.uniform_u;
      float row_val;
      if (a.loss_kind == KGE_LOSS_POSITIVE) {              // model.py:277-279
        const float s = sc[0];
        row_val = log_sigmoid(s);
        if (tid == 0) gg[0] = -0.5f * u * sigmoid(-s);
      } else {
        float zmax = -INFINITY;
        if (a.loss_kind == KGE_LOSS_NEG_ADVERSARIAL) {     // softmax(alpha * s).detach(), model.py:272
          for (int n = tid; n < a.N; n += blockDim.x) zmax = fmaxf(zmax, sc[n] * a.alpha);
          zmax = block_reduce(zmax, scratch, true);
        }
        float zsum = 0.f;
        for (int n = tid; n < a.N; n += blockDim.x) {
          const float e = a.loss_kind == KGE_LOSS_NEG_ADVERSARIAL ? expf(sc[n] * a.alpha - zmax) : 1.f;
          gg[n] = e;
          zsum += e;
        }
        zsum = block_reduce(zsum, scratch, false);
        float acc = 0.f;
        for (int n = tid; n < a.N; n += blockDim.x) {
          const float w = gg[n] / zsum;                    // = 1/N for the uniform case (model.py:275)
          const float s = sc[n];
          acc += w * log_sigmoid(-s);
          gg[n] = 0.5f * u * w * sigmoid(s);
        }
        row_val = block_reduce(acc, scratch, false);
      }
      if (tid == 0) a.row_loss[b] = row_val;
      __syncthreads();
    }
    if (!do_bwd) continue;
    const float *gsrc = a.do_loss ? gg : a.dscore + (int64_t)rl * a.N;

    // ---- phase 3/4: backward over the candidates, k-tiled so dL/dq stays in registers -----------------
    float gmod = 0.f;
    for (int kt = 0; kt < nunits; kt += 32 * kChunks) {
      float acc[kChunks][H][V];
#pragma unroll
      for (int i = 0; i < kChunks; ++i)
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
          for (int j = 0; j < V; ++j) acc[i][h][j] = 0.f;

      for (int n = warp; n < a.N; n += nwarps) {
        int64_t id = cand[n];
        if ((uint64_t)id >= (uint64_t)a.nentity) id = 0;
        const float g = gsrc[n];
        const float go = dsum_of<MODEL>(g, modulus);
        const float *x = a.E + id * a.De;
        float *gx = a.gE + id * a.De;
        float vsum = 0.f;
#pragma unroll
        for (int i = 0; i < kChunks; ++i) {
          const int u = kt + lane + 32 * i;
          if (u < nunits) {
            float x0[V], x1[V], q0[V], q1[V], dx0[V], dx1[V];
            load_global<V>(x0, x + u * V);
            load_shared<V>(q0, q + u * V);
            if constexpr (CPLX) {
              load_global<V>(x1, x + a.d + u * V);
              load_shared<V>(q1, q + a.d + u * V);
            }
#pragma unroll
            for (int j = 0; j < V; ++j) {
              float dq0 = 0.f, dq1 = 0.f, ex0 = 0.f, ex1 = 0.f;
              vsum += op_backward<OP>(q0[j], CPLX ? q1[j] : 0.f, x0[j], CPLX ? x1[j] : 0.f, a.scale, go,
                                      dq0, dq1, ex0, ex1);
              acc[i][0][j] += dq0;
              dx0[j] = ex0;
              if constexpr (CPLX) { acc[i][1][j] += dq1; dx1[j] = ex1; }
            }
            red_global<V>(gx + u * V, dx0);
            if constexpr (CPLX) red_global<V>(gx + a.d + u * V, dx1);
          }
        }
        if constexpr (MODEL == KGE_PROTATE) {
          vsum = warp_sum(vsum);
          gmod += -g * vsum;                               // d/dmodulus of gamma - modulus * sum
        }
      }
      // phase 4: fixed-order fold of the per-warp partial dL/dq into shared memory
      for (int w = 0; w < nwarps; ++w) {
        if (warp == w) {
#pragma unroll
          for (int i = 0; i < kChunks; ++i) {
            const int u = kt + lane + 32 * i;
            if (u < nunits) {
#pragma unroll
              for (int j = 0; j < V; ++j) {
                dq[u * V + j] += acc[i][0][j];
                if constexpr (CPLX) dq[a.d + u * V + j] += acc[i][1][j];
              }
            }
          }
        }
        __syncthreads();
      }
    }

    // ---- phase 5: chain rule into the fixed entity row and the relation row -----------------------------
    float *gF = a.gE + fid * a.De;
    float *gRr = a.gR + rid * a.Dr;
    for (int k = tid; k < a.d; k += blockDim.x) {
      float dF0, dF1, dR0, dR1;
      chain_q<MODEL, HEAD>(F, Rr, dq, k, a.d, a.scale, dF0, dF1, dR0, dR1);
      red_add1(gF + k, dF0);
      red_add1(gRr + k, dR0);
      if constexpr (CPLX) red_add1(gF + a.d + k, dF1);
      if constexpr (MODEL == KGE_COMPLEX) red_add1(gRr + a.d + k, dR1);
    }
    if constexpr (MODEL == KGE_PROTATE) {
      if (lane == 0 && gmod != 0.f && a.gM) red_add1(a.gM, gmod);
    }
  }
}

// ======================================================================================================
// TMA variant: candidate rows are gathered by the bulk-copy engine (cp.async.bulk global -> shared, one
// 1-D copy of the whole D_e*4-byte row per candidate, completion on an mbarrier) into a per-warp double
// buffer.  The bytes in flight are then bounded by shared memory (W warps x 2 slots x row bytes, ~200 KB
// per SM) instead of by registers, which is what the direct-load kernel above is limited by (ncu r1a:
// 68% of issue slots stalled on long-scoreboard with 16 KB in flight per SM).  Phases are the same.
// ======================================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {   // bar: shared-window address
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) { mbar_wait(smem_u32(bar), parity); }
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void bulk_g2s_hint(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
      : "memory");
}

// expect_tx of 2 x `bytes` (NCOPY 2) or `bytes` (NCOPY 1) on `bar`, and the copies src0 -> dst0 [, src1 -> dst1],
// issued by one lane that elect.sync picks from the whole (converged) warp.  Every lane passes the same operands (a
// shuffled id): under elect.sync ptxas moves them to uniform registers once, where a `lane == 0` branch made it wrap
// every copy in a re-election loop (ELECT / R2UR / BRA.U.ANY) for operands it could not prove uniform.
// HINT: the copies carry the L2 cache policy `pol`.
#define KGE_BULK_ELECT_HEAD "{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\n@p mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n"
#define KGE_BULK_ELECT_COPY(D, S) \
  "@p cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [" D "], [" S "], %4, [%0];\n"
#define KGE_BULK_ELECT_COPY_HINT(D, S) \
  "@p cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [" D "], [" S "], %4, [%0], %7;\n"
template <int NCOPY, bool HINT>
__device__ __forceinline__ void bulk_g2s_warp(uint32_t bar, uint32_t dst0, const void *src0, uint32_t dst1,
                                              const void *src1, uint32_t bytes, uint64_t pol = 0) {
  static_assert(NCOPY == 1 || NCOPY == 2, "one or two copies");
  if constexpr (HINT && NCOPY == 2)
    asm volatile(KGE_BULK_ELECT_HEAD KGE_BULK_ELECT_COPY_HINT("%2", "%3") KGE_BULK_ELECT_COPY_HINT("%5", "%6") "}\n"
                 ::"r"(bar), "r"(bytes * NCOPY), "r"(dst0), "l"(src0), "r"(bytes), "r"(dst1), "l"(src1), "l"(pol) : "memory");
  else if constexpr (HINT)
    asm volatile(KGE_BULK_ELECT_HEAD KGE_BULK_ELECT_COPY_HINT("%2", "%3") "}\n"
                 ::"r"(bar), "r"(bytes * NCOPY), "r"(dst0), "l"(src0), "r"(bytes), "r"(dst1), "l"(src1), "l"(pol) : "memory");
  else if constexpr (NCOPY == 2)
    asm volatile(KGE_BULK_ELECT_HEAD KGE_BULK_ELECT_COPY("%2", "%3") KGE_BULK_ELECT_COPY("%5", "%6") "}\n"
                 ::"r"(bar), "r"(bytes * NCOPY), "r"(dst0), "l"(src0), "r"(bytes), "r"(dst1), "l"(src1), "l"(pol) : "memory");
  else
    asm volatile(KGE_BULK_ELECT_HEAD KGE_BULK_ELECT_COPY("%2", "%3") "}\n"
                 ::"r"(bar), "r"(bytes * NCOPY), "r"(dst0), "l"(src0), "r"(bytes), "r"(dst1), "l"(src1), "l"(pol) : "memory");
}
#undef KGE_BULK_ELECT_HEAD
#undef KGE_BULK_ELECT_COPY
#undef KGE_BULK_ELECT_COPY_HINT

template <int MODEL, bool HEAD>
__global__ void __launch_bounds__(512, 1) row_kernel_tma(const RowArgs a) {
  constexpr int OP = op_of(MODEL, HEAD);
  constexpr bool CPLX = op_is_complex(OP);
  constexpr int H = CPLX ? 2 : 1;
  constexpr int V = 4;
  constexpr int CH = CPLX ? 8 : 16;            // units per lane: 64 accumulator registers either way
  extern __shared__ __align__(128) float smem[];
  const int Dq = a.De;
  const int Dq4 = (Dq + 3) & ~3;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  // layout: [slots: nwarps x 2 x De | q | dq | sc | gg | scratch(32) | mbarriers]; every pointer is derived from
  // `smem` by element offsets so that the compiler keeps the shared address space (LDS, not generic LD)
  float *slot0 = smem + (size_t)(2 * warp) * a.De, *slot1 = slot0 + a.De;
  float *q = smem + (size_t)(2 * nwarps) * a.De;
  float *dq = q + Dq4;
  float *sc = dq + Dq4;
  float *gg = sc + (a.do_loss ? a.N : 0);
  float *scratch = gg + (a.do_loss ? a.N : 0);
  uint64_t *bars = reinterpret_cast<uint64_t *>(scratch + 32);
  const uint32_t rowbytes = (uint32_t)a.De * 4u;
  uint64_t *bar0 = bars + 2 * warp, *bar1 = bar0 + 1;
  uint32_t par0 = 0, par1 = 0;
  int64_t id0 = 0, id1 = 0;

  const int nunits = a.d / V;                  // <= 32 * CH (host)
  const float modulus = MODEL == KGE_PROTATE ? __ldg(a.modulus) : 1.f;
  const bool do_bwd = a.gE != nullptr;

  if (lane == 0) { mbar_init(bar0, 1); mbar_init(bar1, 1); }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  for (int rl = blockIdx.x; rl < a.row_count; rl += gridDim.x) {
    const int64_t b = a.row_begin + rl;
    int64_t hid = a.positive[b * 3 + 0], rid = a.positive[b * 3 + 1], tidx = a.positive[b * 3 + 2];
    int64_t fid = HEAD ? tidx : hid;
    if ((uint64_t)fid >= (uint64_t)a.nentity || (uint64_t)rid >= (uint64_t)a.nrelation) {
      if (tid == 0 && a.err) *a.err = 1;
      fid = 0; rid = 0;
    }
    const float *F = a.E + fid * a.De;
    const float *Rr = a.R + rid * a.Dr;
    const int64_t *cand = a.cand + b * a.cand_stride;

    // issue the bulk copy of candidate n into this warp's slot s (all lanes run it; lane 0 talks to the engine)
    auto issue = [&](int s, int n) {
      int64_t id = cand[n];
      if ((uint64_t)id >= (uint64_t)a.nentity) { if (lane == 0 && a.err) *a.err = 1; id = 0; }
      if (s) id1 = id; else id0 = id;
      if (lane == 0) {
        uint64_t *bar = s ? bar1 : bar0;
        mbar_expect_tx(bar, rowbytes);
        bulk_g2s(s ? slot1 : slot0, a.E + id * a.De, rowbytes, bar);
      }
    };
    // first two candidates of phase 1 (or of phase 3 for the backward-only call) overlap the q build
    if (warp < a.N) issue(0, warp);
    if (warp + nwarps < a.N) issue(1, warp + nwarps);

    // ---- phase 0: query vector -------------------------------------------------------------------
    for (int k = tid; k < a.d; k += blockDim.x) {
      build_q<MODEL, HEAD>(F, Rr, k, a.d, a.scale, q);
      dq[k] = 0.f;
      if (CPLX) dq[a.d + k] = 0.f;
    }
    __syncthreads();

    // ---- phase 1: scores -------------------------------------------------------------------------
    const bool do_fwd = a.do_loss || a.score_out;
    if (do_fwd) {
      int it = 0;
      for (int n = warp; n < a.N; n += nwarps, ++it) {
        const int s = it & 1;
        if (s) { mbar_wait(bar1, par1); par1 ^= 1; } else { mbar_wait(bar0, par0); par0 ^= 1; }
        const float *x = s ? slot1 : slot0;
        float part = 0.f;
#pragma unroll
        for (int i = 0; i < CH; ++i) {
          const int u = lane + 32 * i;
          if (u < nunits) {
            float x0[V], x1[V], q0[V], q1[V];
            load_shared<V>(x0, x + u * V);
            load_shared<V>(q0, q + u * V);
            if constexpr (CPLX) {
              load_shared<V>(x1, x + a.d + u * V);
              load_shared<V>(q1, q + a.d + u * V);
            }
#pragma unroll
            for (int j = 0; j < V; ++j)
              part += op_forward<OP>(q0[j], CPLX ? q1[j] : 0.f, x0[j], CPLX ? x1[j] : 0.f, a.scale);
          }
        }
        __syncwarp();                                   // every lane is done reading the slot
        if (n + 2 * nwarps < a.N) issue(s, n + 2 * nwarps);
        part = warp_sum(part);
        const float sv = finish_score<MODEL>(part, a.gamma, modulus);
        if (lane == 0) {
          if (a.do_loss) sc[n] = sv;
          if (a.score_out) a.score_out[(int64_t)rl * a.N + n] = sv;
        }
      }
      if (do_bwd) {                                     // restart the ring for phase 3 while the loss is computed
        if (warp < a.N) issue(0, warp);
        if (warp + nwarps < a.N) issue(1, warp + nwarps);
      }
    }
    if (!a.do_loss && !do_bwd) { __syncthreads(); continue; }

    // ---- phase 2: loss of this row (model.py:270-288) and dL/ds ---------------------------------------
    if (a.do_loss) {
      __syncthreads();
      const float u = a.weight ? a.weight[b] / a.wsum[0] : a.uniform_u;
      float row_val;
      if (a.loss_kind == KGE_LOSS_POSITIVE) {
        const float sv = sc[0];
        row_val = log_sigmoid(sv);
        if (tid == 0) gg[0] = -0.5f * u * sigmoid(-sv);
      } else {
        float zmax = -INFINITY;
        if (a.loss_kind == KGE_LOSS_NEG_ADVERSARIAL) {
          for (int n = tid; n < a.N; n += blockDim.x) zmax = fmaxf(zmax, sc[n] * a.alpha);
          zmax = block_reduce(zmax, scratch, true);
        }
        float zsum = 0.f;
        for (int n = tid; n < a.N; n += blockDim.x) {
          const float e = a.loss_kind == KGE_LOSS_NEG_ADVERSARIAL ? expf(sc[n] * a.alpha - zmax) : 1.f;
          gg[n] = e;
          zsum += e;
        }
        zsum = block_reduce(zsum, scratch, false);
        float acc = 0.f;
        for (int n = tid; n < a.N; n += blockDim.x) {
          const float w = gg[n] / zsum;
          const float sv = sc[n];
          acc += w * log_sigmoid(-sv);
          gg[n] = 0.5f * u * w * sigmoid(sv);
        }
        row_val = block_reduce(acc, scratch, false);
      }
      if (tid == 0) a.row_loss[b] = row_val;
      __syncthreads();
    }
    if (!do_bwd) continue;
    const float *gsrc = a.do_loss ? gg : a.dscore + (int64_t)rl * a.N;

    // ---- phase 3: backward over the candidates; dL/dq stays in registers ------------------------------------
    float gmod = 0.f;
    float acc[CH][H][V];
#pragma unroll
    for (int i = 0; i < CH; ++i)
#pragma unroll
      for (int h = 0; h < H; ++h)
#pragma unroll
        for (int j = 0; j < V; ++j) acc[i][h][j] = 0.f;
    {
      int it = 0;
      for (int n = warp; n < a.N; n += nwarps, ++it) {
        const int s = it & 1;
        if (s) { mbar_wait(bar1, par1); par1 ^= 1; } else { mbar_wait(bar0, par0); par0 ^= 1; }
        const float *x = s ? slot1 : slot0;
        const int64_t id = s ? id1 : id0;
        const float g = gsrc[n];
        const float go = dsum_of<MODEL>(g, modulus);
        float *gx = a.gE + id * a.De;
        float vsum = 0.f;
#pragma unroll
        for (int i = 0; i < CH; ++i) {
          const int u = lane + 32 * i;
          if (u < nunits) {
            float x0[V], x1[V], q0[V], q1[V], dx0[V], dx1[V];
            load_shared<V>(x0, x + u * V);
            load_shared<V>(q0, q + u * V);
            if constexpr (CPLX) {
              load_shared<V>(x1, x + a.d + u * V);
              load_shared<V>(q1, q + a.d + u * V);
            }
#pragma unroll
            for (int j = 0; j < V; ++j) {
              float dq0 = 0.f, dq1 = 0.f, ex0 = 0.f, ex1 = 0.f;
              vsum += op_backward<OP>(q0[j], CPLX ? q1[j] : 0.f, x0[j], CPLX ? x1[j] : 0.f, a.scale, go,
                                      dq0, dq1, ex0, ex1);
              acc[i][0][j] += dq0;
              dx0[j] = ex0;
              if constexpr (CPLX) { acc[i][1][j] += dq1; dx1[j] = ex1; }
            }
            red_global<V>(gx + u * V, dx0);
            if constexpr (CPLX) red_global<V>(gx + a.d + u * V, dx1);
          }
        }
        __syncwarp();
        if (n + 2 * nwarps < a.N) issue(s, n + 2 * nwarps);
        if constexpr (MODEL == KGE_PROTATE) {
          vsum = warp_sum(vsum);
          gmod += -g * vsum;
        }
      }
    }
    // ---- phase 4: fixed-order fold of the per-warp partial dL/dq into shared memory -----------------------
    for (int w = 0; w < nwarps; ++w) {
      if (warp == w) {
#pragma unroll
        for (int i = 0; i < CH; ++i) {
          const int u = lane + 32 * i;
          if (u < nunits) {
#pragma unroll
            for (int j = 0; j < V; ++j) {
              dq[u * V + j] += acc[i][0][j];
              if constexpr (CPLX) dq[a.d + u * V + j] += acc[i][1][j];
            }
          }
        }
      }
      __syncthreads();
    }
    // ---- phase 5: chain rule into the fixed entity row and the relation row -----------------------------
    float *gF = a.gE + fid * a.De;
    float *gRr = a.gR + rid * a.Dr;
    for (int k = tid; k < a.d; k += blockDim.x) {
      float dF0, dF1, dR0, dR1;
      chain_q<MODEL, HEAD>(F, Rr, dq, k, a.d, a.scale, dF0, dF1, dR0, dR1);
      red_add1(gF + k, dF0);
      red_add1(gRr + k, dR0);
      if constexpr (CPLX) red_add1(gF + a.d + k, dF1);
      if constexpr (MODEL == KGE_COMPLEX) red_add1(gRr + a.d + k, dR1);
    }
    if constexpr (MODEL == KGE_PROTATE) {
      if (lane == 0 && gmod != 0.f && a.gM) red_add1(a.gM, gmod);
    }
    __syncthreads();                                    // q / dq are rebuilt by the next row
  }
}

}  // namespace kge
