// kge_eval_gemm.cu -- tcgen05 (5th-gen tensor core) all-entity scoring for the dot-product models
// (DistMult model.py:175-182, ComplEx model.py:184-199) in test_step, with ranks that stay bit-exact.
//
// For these two models  score(q, j) = <qvec_q, E_j>  is a real [Q, D_e] x [D_e, nentity] contraction -- the one
// dense GEMM of the path.  fp32 has no tensor-core kind, so every operand is split once into two TF32-exact
// pieces  x = hi + lo (+ r, |r| <= 2^-20 |x|)  and the kernel accumulates  hi*hi + hi*lo + lo*hi  (3xTF32) in
// fp32 in tensor memory.  That result is only an *approximation* of the canonical fp32 score that defines the
// ranks (DESIGN.md section 4), with a rigorous bound  |approx - canonical| <= eps_qj = kBand * |q| * |E_j|.
// The epilogue therefore classifies each (query, entity):
//      approx - eps > s_pos  -> certainly ranked above the positive: count it
//      approx + eps < s_pos  -> certainly below: ignore
//      otherwise             -> ambiguous: append (q, j) to a list
// and rescore_pairs_kernel re-scores the short ambiguous list with the canonical exact op sequence.  Counts (and
// ranks) are therefore identical to the exact SIMT kernel's, whatever the tensor core's internal rounding is.
//
// Kernel anatomy (one CTA per 128-query tile, looping over 128-entity tiles):
//   warp 0   TMA producer: per 32-wide k-block FOUR cp.async.bulk.tensor 2-D tiles (SWIZZLE_128B: Q_hi, Q_lo of 128 rows
//            x 32 fp32, E_hi, E_lo of 256 rows x 32 fp32) into one 96 KB stage of a 2-stage ring, mbarrier complete_tx
//   warp 1   MMA issuer: one elected lane issues 12 tcgen05.mma.cta_group::1.kind::tf32 (M=128, N=256, K=8) per stage
//            -- hi*hi, hi*lo, lo*hi on the same four tiles -- accumulating in TMEM; tcgen05.commit frees ring slots /
//            publishes tiles.  (Round 1 streamed the three products as separate passes over two-tile stages: 32 KB of
//            operands per 4 128x128x8 MMAs = 120 B/clk per SM, more than L2 delivers; ncu r1g: tensor pipe 52 % active.
//            Four tiles with a 256-wide entity tile feed the equivalent of 24 such MMAs from 96 KB: 60 B/clk.)
//   warp 2   TMEM allocator (512 columns = two 128 x 256 accumulator buffers)
//   warps 4-7  epilogue: tcgen05.ld 32x32b (lane = query row), band test, filter bitmap, counts, ambiguous list
#include <cuda.h>

#include "kge_rows.cuh"

namespace kge {

constexpr int GM = 128, GN = 256, GK = 32, GSTAGES = 2, GTHREADS = 256;
constexpr uint32_t kTileBytes = GM * GK * 4;                  // 16 KB per query tile (128 rows x 32 fp32)
constexpr uint32_t kTileBytesB = GN * GK * 4;                 // 32 KB per entity tile (256 rows x 32 fp32)
constexpr uint32_t kStageBytes = 2 * kTileBytes + 2 * kTileBytesB;   // Q_hi | Q_lo | E_hi | E_lo = 96 KB
// eps = band * |q| * |e| with band = kBandSplit + kBandPerKBlock * (number of 32-wide k-blocks issued):
//   kBandSplit      operand residuals (3 * 2^-20), the dropped lo*lo term, and the rounding of the canonical fp32 sum
//   kBandPerKBlock  4 tcgen05.mma per k-block, each assumed to add at most 2^-22 of the magnitude bound |q||e| when it
//                   folds 8 exact products into the fp32 accumulator (truncating accumulate with a guard bit)
constexpr float kBandSplit = 1.0e-5f, kBandPerKBlock = 9.6e-7f;

struct GemmArgs {
  const float *pos_score;        // [Q] canonical score of the positive
  const float *qnorm, *enorm;    // [Q], [nentity] euclidean norms
  const int64_t *queries;        // [Q,3]
  const uint32_t *filter_bits;   // [Q, words]
  int32_t *counts;               // [Q]
  int2 *amb;                     // ambiguous (q, j) pairs
  int *amb_count;                // [0] = number appended, [1] = overflow flag
  int amb_capacity;
  int Q, pos_col, words;
  int64_t nentity, ent_begin, ent_end;
  int K;                         // contraction length (entity_dim)
  float band;
  float *approx_out;             // tests: [Q, nentity] dump of the tensor-core approximations (or NULL)
};

// ---- PTX wrappers -------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mb_init(uint64_t *b, uint32_t n) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(b)), "r"(n) : "memory");
}
__device__ __forceinline__ void mb_expect(uint64_t *b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_arrive(uint64_t *b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(b)) : "memory");
}
__device__ __forceinline__ void mb_wait(uint64_t *b, uint32_t parity) {
  uint32_t done = 0;
  const long long t0 = clock64();
  while (!done) {
    asm volatile(
        "{\n.reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(done)
        : "r"(s32(b)), "r"(parity)
        : "memory");
    if (!done && clock64() - t0 > 4000000000ll) __trap();   // ~2 s: a broken pipeline fails loudly, it never hangs
  }
}
__device__ __forceinline__ void tma_2d(void *dst, const CUtensorMap *map, int c0, int c1, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          s32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(s32(bar))
      : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n.reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, SWIZZLE_128B operand tile (rows of 128 B, 8-row groups 1024 B apart): cute::UMMA::SmemDescriptor
__device__ __forceinline__ uint64_t smem_desc(const void *tile) {
  uint64_t d = 0;
  d |= (uint64_t)((s32(tile) >> 4) & 0x3FFF);          // start address, bits [0,14)
  d |= (uint64_t)1 << 16;                              // leading byte offset (unused for swizzled K-major) = 1
  d |= (uint64_t)(1024 >> 4) << 32;                    // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                              // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                              // layout type SWIZZLE_128B
  return d;
}
// cute::UMMA::InstrDescriptor for kind::tf32, fp32 accumulate, both operands K-major
__host__ __device__ constexpr uint32_t instr_desc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// STATS: a.counts is the [Q, KGE_RANK_STATS] table of kge_eval_gemm_count_rank_stats; filtered columns are classified too
// (their approximation against the band), and the kernel adds counters [0] (unfiltered, greater) and [3] (greater).
template <bool STATS>
__global__ void __launch_bounds__(GTHREADS, 1)
gemm_count_kernel(const __grid_constant__ CUtensorMap tmQhi, const __grid_constant__ CUtensorMap tmQlo,
                  const __grid_constant__ CUtensorMap tmEhi, const __grid_constant__ CUtensorMap tmElo,
                  const GemmArgs a) {
  extern __shared__ __align__(1024) uint8_t gsm_raw[];
  uint8_t *gsm = gsm_raw + ((1024u - (s32(gsm_raw) & 1023u)) & 1023u);     // SWIZZLE_128B tiles need 1024-B alignment
  uint8_t *tiles = gsm;                                         // [GSTAGES][Q_hi | Q_lo | E_hi | E_lo]
  uint64_t *full = reinterpret_cast<uint64_t *>(gsm + GSTAGES * kStageBytes);
  uint64_t *empty = full + GSTAGES;
  uint64_t *tfull = empty + GSTAGES;                            // [2] accumulator ready
  uint64_t *tempty = tfull + 2;                                 // [2] accumulator drained
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  float *enorm_s = reinterpret_cast<float *>(tmem_slot + 4);    // [2][GN]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * GM;
  const int64_t ntiles_all = (a.ent_end - a.ent_begin + GN - 1) / GN;
  const int nkb = (a.K + GK - 1) / GK;                          // k-blocks; each carries hi*hi, hi*lo, lo*hi

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < GSTAGES; ++i) { mb_init(full + i, 1); mb_init(empty + i, 1); }
    for (int i = 0; i < 2; ++i) { mb_init(tfull + i, 1); mb_init(tempty + i, 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQhi) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQlo) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmEhi) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmElo) : "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(s32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t jt = blockIdx.y; jt < ntiles_all; jt += gridDim.y) {
        const int j0 = (int)(a.ent_begin + jt * GN);
        for (int kb = 0; kb < nkb; ++kb) {
          const int kk = kb * GK;
          uint8_t *t = tiles + (size_t)stage * kStageBytes;
          mb_wait(empty + stage, phase ^ 1);
          mb_expect(full + stage, kStageBytes);
          tma_2d(t, &tmQhi, kk, q0, full + stage);
          tma_2d(t + kTileBytes, &tmQlo, kk, q0, full + stage);
          tma_2d(t + 2 * kTileBytes, &tmEhi, kk, j0, full + stage);
          tma_2d(t + 2 * kTileBytes + kTileBytesB, &tmElo, kk, j0, full + stage);
          if (++stage == GSTAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer =======================================
    if (lane == 0) {
      constexpr uint32_t idesc = instr_desc_tf32(GM, GN);
      int stage = 0;
      uint32_t phase = 0;
      int tile_it = 0;
      for (int64_t jt = blockIdx.y; jt < ntiles_all; jt += gridDim.y, ++tile_it) {
        const int as = tile_it & 1;
        mb_wait(tempty + as, ((tile_it >> 1) & 1) ^ 1);         // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * GN;
        for (int kb = 0; kb < nkb; ++kb) {
          mb_wait(full + stage, phase);
          tc_fence_after();
          const uint8_t *t = tiles + (size_t)stage * kStageBytes;
          const uint64_t qhi = smem_desc(t), qlo = smem_desc(t + kTileBytes);
          const uint64_t ehi = smem_desc(t + 2 * kTileBytes), elo = smem_desc(t + 2 * kTileBytes + kTileBytesB);
#pragma unroll
          for (int k = 0; k < GK / 8; ++k) {                    // UMMA_K = 8 for tf32: advance 32 B inside the swizzle atom
            const uint64_t o = (uint64_t)(k * 2);
            umma_tf32(d_tmem, qhi + o, ehi + o, idesc, (kb | k) ? 1u : 0u);
            umma_tf32(d_tmem, qhi + o, elo + o, idesc, 1u);
            umma_tf32(d_tmem, qlo + o, ehi + o, idesc, 1u);
          }
          umma_commit(empty + stage);                           // slot free once these MMAs have read it
          if (++stage == GSTAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(tfull + as);                                // accumulator complete
      }
    }
  } else if (warp >= 4) {
    // ===================================== epilogue ========================================
    const int ew = warp - 4;                                    // TMEM lanes [32 ew, 32 ew + 32)
    const int row = ew * 32 + lane;
    const int qi = q0 + row;
    const bool qvalid = qi < a.Q;
    const float sp = qvalid ? a.pos_score[qi] : 0.f;
    const float qn = qvalid ? a.qnorm[qi] * a.band : 0.f;
    const int64_t pid = qvalid ? a.queries[(int64_t)qi * 3 + a.pos_col] : -1;
    const uint32_t *frow = a.filter_bits + (int64_t)(qvalid ? qi : 0) * a.words;
    int count = 0;
    [[maybe_unused]] int count_raw = 0;
    int tile_it = 0;
    for (int64_t jt = blockIdx.y; jt < ntiles_all; jt += gridDim.y, ++tile_it) {
      const int as = tile_it & 1;
      const int64_t j0 = a.ent_begin + jt * GN;
      // entity norms of this tile (threads 128..255 -> GN values), visible after the named barrier
      for (int t = threadIdx.x - 128; t < GN; t += 128) {
        const int64_t j = j0 + t;
        enorm_s[as * GN + t] = j < a.ent_end ? a.enorm[j] : 0.f;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      mb_wait(tfull + as, (tile_it >> 1) & 1);
      tc_fence_after();
      uint32_t amask[GN / 32];                                  // ambiguous columns of this row, one word per chunk
#pragma unroll
      for (int c = 0; c < GN / 32; ++c) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(as * GN + c * 32);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,"
            "%28,%29,%30,%31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
              "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
              "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
              "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        uint32_t am = 0;
        if (qvalid) {
          const int64_t jb = j0 + c * 32;
          const uint32_t fw = jb < a.ent_end ? frow[jb >> 5] : 0u;    // tiles are 32-aligned: one bitmap word
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int64_t j = jb + i;
            if (a.approx_out && j < a.ent_end) a.approx_out[(int64_t)qi * a.nentity + j] = __uint_as_float(v[i]);
            if (j >= a.ent_end || j == pid || (!STATS && ((fw >> i) & 1u))) continue;
            const float s = __uint_as_float(v[i]);
            const float eps = qn * enorm_s[as * GN + c * 32 + i];
            if (s - eps > sp) {
              if constexpr (STATS) {
                count += !((fw >> i) & 1u);
                ++count_raw;
              } else {
                ++count;
              }
            } else if (s + eps >= sp) am |= 1u << i;           // cannot be decided from the approximation
          }
        }
        amask[c] = am;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mb_arrive(tempty + as);                    // 4 epilogue warps -> accumulator free
      // one reservation per warp and tile in the ambiguous list, then every row writes its own pairs
      int mine = 0;
#pragma unroll
      for (int c = 0; c < GN / 32; ++c) mine += __popc(amask[c]);
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const int total = __shfl_sync(0xffffffffu, incl, 31);
      if (total) {
        int base = 0;
        if (lane == 0) base = atomicAdd(a.amb_count, total);
        base = __shfl_sync(0xffffffffu, base, 0) + incl - mine;
#pragma unroll
        for (int c = 0; c < GN / 32; ++c) {
          uint32_t am = amask[c];
          while (am) {
            const int i = __ffs(am) - 1;
            am &= am - 1;
            if (base < a.amb_capacity) a.amb[base] = make_int2(qi, (int)(j0 + c * 32 + i));
            else a.amb_count[1] = 1;
            ++base;
          }
        }
      }
    }
    if constexpr (STATS) {
      if (qvalid && count) atomicAdd(a.counts + (int64_t)qi * KGE_RANK_STATS, count);
      if (qvalid && count_raw) atomicAdd(a.counts + (int64_t)qi * KGE_RANK_STATS + 3, count_raw);
    } else {
      if (qvalid && count) atomicAdd(a.counts + qi, count);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// ---- operand preparation -----------------------------------------------------------------------------------
// x = hi + lo + r with hi, lo exactly representable in TF32 (low 13 mantissa bits zero), |r| <= 2^-20 |x|.
__global__ void split_tf32_kernel(const float *__restrict__ x, int64_t rows, int cols, float *__restrict__ hi,
                                  float *__restrict__ lo, float *__restrict__ norm) {
  for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
    float acc = 0.f;
    for (int c = threadIdx.x; c < cols; c += blockDim.x) {
      const float v = x[r * cols + c];
      const float h = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
      const float l = __uint_as_float(__float_as_uint(v - h) & 0xFFFFE000u);
      hi[r * cols + c] = h;
      lo[r * cols + c] = l;
      acc += v * v;
    }
    __shared__ float sh[8];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i];
      norm[r] = sqrtf(t) * 1.0001f;                          // rounded up: the band must never be too small
    }
    __syncthreads();
  }
}

int launch_rescore_pairs(bool cplx, const void *amb, const int *amb_count, int capacity, const float *qvec,
                         const float *E, int d, int De, const float *pos_score, const int64_t *queries, int pos_col,
                         int32_t *counts, cudaStream_t st, const uint32_t *filter_bits = nullptr,
                         int words = 0);                                          // kge_eval.cu (exact op sequence)

// ---- host ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_map(CUtensorMap *map, const float *base, int64_t rows, int64_t cols, int box_rows) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    KGE_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    KGE_REQUIRE(p && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled is not available in this driver");
    fn = (EncodeTiledFn)p;
  }
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  const cuuint32_t box[2] = {GK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)base, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  KGE_REQUIRE(rc == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d", (int)rc);
  return KGE_OK;
}

}  // namespace kge

using namespace kge;

extern "C" int kge_eval_gemm_supported(const kge_model_t *m) {
  if (!m) return 0;
  return (m->model == KGE_DISTMULT || m->model == KGE_COMPLEX) && m->entity_dim % 4 == 0 &&
         (((uintptr_t)m->entity) & 15) == 0 && m->nentity < (1ll << 31);
}

extern "C" float kge_eval_gemm_band(int64_t entity_dim) {
  return kBandSplit + kBandPerKBlock * (float)(3 * ((entity_dim + GK - 1) / GK));
}

extern "C" int kge_eval_gemm_split(const float *x, int64_t rows, int64_t cols, float *hi, float *lo, float *norm,
                                   void *stream) {
  KGE_REQUIRE(x && hi && lo && norm && rows > 0 && cols > 0, "bad arguments");
  const int grid = (int)(rows < 148 * 16 ? rows : 148 * 16);
  split_tf32_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, rows, (int)cols, hi, lo, norm);
  KGE_CUDA_OK(cudaGetLastError());
  return KGE_OK;
}

static int gemm_count_impl(const kge_model_t *m, int mode, const float *qvec, const float *qhi, const float *qlo,
                           const float *qnorm, const int64_t *queries, int64_t Q, const float *pos_score,
                           const uint32_t *filter_bits, const float *ehi, const float *elo, const float *enorm,
                           int64_t ent_begin, int64_t ent_end, int32_t *counts, void *amb_pairs, int64_t amb_capacity,
                           int32_t *amb_count, float *approx_scores_out, void *stream, bool stats) {
  int rc = check_model(m);
  if (rc) return rc;
  KGE_REQUIRE(kge_eval_gemm_supported(m), "the tcgen05 path serves DistMult / ComplEx with 16-byte aligned rows");
  KGE_REQUIRE(mode == KGE_HEAD_BATCH || mode == KGE_TAIL_BATCH, "negative batch mode %d not supported", mode);
  KGE_REQUIRE(qvec && qhi && qlo && qnorm && queries && pos_score && filter_bits && ehi && elo && enorm && counts &&
                  amb_pairs && amb_count && amb_capacity > 0,
              "null pointer");
  KGE_REQUIRE(ent_begin >= 0 && ent_begin <= ent_end && ent_end <= m->nentity && ent_begin % 32 == 0,
              "entity slice must start on a multiple of 32");
  if (Q <= 0 || ent_begin == ent_end) return KGE_OK;
  DeviceGuard device_guard;
  if ((rc = device_guard.enter(m->device))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t K = m->entity_dim;
  CUtensorMap tQhi, tQlo, tEhi, tElo;
  if ((rc = make_map(&tQhi, qhi, Q, K, GM))) return rc;
  if ((rc = make_map(&tQlo, qlo, Q, K, GM))) return rc;
  if ((rc = make_map(&tEhi, ehi, m->nentity, K, GN))) return rc;
  if ((rc = make_map(&tElo, elo, m->nentity, K, GN))) return rc;
  GemmArgs a{};
  a.pos_score = pos_score; a.qnorm = qnorm; a.enorm = enorm; a.queries = queries; a.filter_bits = filter_bits;
  a.counts = counts; a.amb = (int2 *)amb_pairs; a.amb_count = amb_count; a.amb_capacity = (int)amb_capacity;
  a.Q = (int)Q; a.pos_col = mode == KGE_HEAD_BATCH ? 0 : 2; a.words = (int)((m->nentity + 31) / 32);
  a.nentity = m->nentity; a.ent_begin = ent_begin; a.ent_end = ent_end; a.K = (int)K;
  a.band = kge_eval_gemm_band(K);
  a.approx_out = approx_scores_out;
  KGE_CUDA_OK(cudaMemsetAsync(amb_count, 0, 2 * sizeof(int), st));
  const size_t smem = GSTAGES * kStageBytes + (2 * GSTAGES + 4) * 8 + 16 + 2 * GN * 4 + 1024;
  auto kernel = stats ? gemm_count_kernel<true> : gemm_count_kernel<false>;
  KGE_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int qtiles = (int)((Q + GM - 1) / GM);
  const int64_t jtiles = (ent_end - ent_begin + GN - 1) / GN;
  int ysplit = 148 / qtiles;                                      // one wave: at most 148 CTAs (one per SM)
  if (ysplit > jtiles) ysplit = (int)jtiles;
  if (ysplit < 1) ysplit = 1;
  kernel<<<dim3(qtiles, ysplit), GTHREADS, smem, st>>>(tQhi, tQlo, tEhi, tElo, a);
  KGE_CUDA_OK(cudaGetLastError());
  const bool cplx = m->model == KGE_COMPLEX;
  const int d = cplx ? (int)(K / 2) : (int)K;
  if ((rc = launch_rescore_pairs(cplx, a.amb, amb_count, a.amb_capacity, qvec, m->entity, d, (int)K, pos_score, queries,
                                 a.pos_col, counts, st, stats ? filter_bits : nullptr, a.words)))
    return rc;
  return KGE_OK;
}

extern "C" int kge_eval_gemm_count_ranks(const kge_model_t *m, int mode, const float *qvec, const float *qhi,
                                         const float *qlo, const float *qnorm, const int64_t *queries, int64_t Q,
                                         const float *pos_score, const uint32_t *filter_bits, const float *ehi,
                                         const float *elo, const float *enorm, int64_t ent_begin, int64_t ent_end,
                                         int32_t *counts, void *amb_pairs, int64_t amb_capacity, int32_t *amb_count,
                                         float *approx_scores_out, void *stream) {
  return gemm_count_impl(m, mode, qvec, qhi, qlo, qnorm, queries, Q, pos_score, filter_bits, ehi, elo, enorm, ent_begin,
                         ent_end, counts, amb_pairs, amb_capacity, amb_count, approx_scores_out, stream, false);
}

extern "C" int kge_eval_gemm_count_rank_stats(const kge_model_t *m, int mode, const float *qvec, const float *qhi,
                                              const float *qlo, const float *qnorm, const int64_t *queries, int64_t Q,
                                              const float *pos_score, const uint32_t *filter_bits, const float *ehi,
                                              const float *elo, const float *enorm, int64_t ent_begin, int64_t ent_end,
                                              int32_t *stats, void *amb_pairs, int64_t amb_capacity,
                                              int32_t *amb_count, void *stream) {
  return gemm_count_impl(m, mode, qvec, qhi, qlo, qnorm, queries, Q, pos_score, filter_bits, ehi, elo, enorm, ent_begin,
                         ent_end, stats, amb_pairs, amb_capacity, amb_count, nullptr, stream, true);
}
