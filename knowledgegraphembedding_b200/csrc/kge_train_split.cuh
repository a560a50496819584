// kge_train_split.cuh -- single-read train path: row-major forward + dL/dq, entity-major dL/dx (+ Adam).
//
// The two-sweep row kernel (kge_train_kernels.cuh) reads every candidate row twice and scatters dL/dx with
// 2.1 GB of atomics into a gradient table that does not fit L2 next to the entity table (ncu r1b:
// 4.78 GB of DRAM traffic, L2 hit 33 %).  This path reads each candidate row ONCE from global memory:
//
//   row_kernel_split   (persistent, one CTA per SM walking its positive rows, TMA ring per warp)
//       per candidate: one sweep over the shared-memory slot -> score and u = d(value)/dq, both in registers;
//       then acc += coef * u with a *deferred* softmax normalisation (each warp keeps a running max M_w of
//       alpha*s and rescales its accumulator when the max grows, exactly like an online softmax); after the
//       row's loss is known the accumulators are brought to the common max, folded, scaled by  -/+ u/(2 Z)
//       and pushed through the chain rule.  It also writes q[b] and g[b,n] = dL/ds to a workspace and
//       histograms the candidate ids.
//   scan_tiles + scan_apply / scatter_pairs   counting sort of the (b,n) pairs by candidate entity
//   entity_kernel      (one warp per (entity, half row), dynamic queue) the entity row x_e sits in registers; the
//       q rows of its pairs (8 MB table, L2 resident) arrive through a TMA double buffer; dL/dx is summed in
//       registers.  Then either the sum is added to the gradient row once (no atomics), or -- fused optimizer,
//       kge_train_rows_adam -- the gradient rows of the positive triples arrive through the same buffer, and the warp
//       applies torch.optim.Adam to its slice of the entity row in place: the dense entity gradient never exists.
//
// DRAM traffic drops from ~1.1 x A to the first touch of the entity table plus (fused optimizer) one read of the two
// moment tables and one write of tables and moments; the passes are shared-memory-bandwidth / issue bound.
#pragma once
#include "kge_train_kernels.cuh"

namespace kge {

// NCH = 128-float chunks per half row (4, 8 or 16): the halves of a row sit at a fixed padded stride DP = 128 * NCH
// floats in every shared-memory slot and in q, the pad is zero (and stays zero: every element op maps (q, x) = (0, 0) to
// value 0 and u 0), so the per-lane loops over the row have compile-time trip counts and immediate address offsets --
// no bounds guards, no divergence bookkeeping (the guarded version spent 11 % of its instructions on them).
//
// VAR picks where a lane keeps u = d(value)/dq between the score sweep and the accumulate step, and where q lives:
//   0  u parked in the slot (STS + second LDS pass + a proxy fence per candidate), q in shared memory   [round 1]
//   1  u in registers, q in shared memory
//   2  u and q in registers: per candidate the only shared-memory traffic is one read of the row
//   3  like 2, but TWO warps share a candidate row (each covers half of the 128-float chunks): a third of the
//      registers per thread less, so 12 warps (6 pairs) instead of 8 are resident to cover the fixed-latency stalls that
//      ncu r2a shows for variant 2 (36 % issue-slot use with 2 warps per scheduler); the halves of the score meet through
//      one shared-memory word per warp and one 64-thread named barrier per candidate
//   4  like 3 with 16 warps (8 pairs) at 128 registers
// ncu r1l showed variant 0 bound by shared-memory bandwidth (40 KB moved per 8 KB candidate row: TMA write, x, q,
// u out, u back); variants 1 / 2 move 24 / 16 KB.  The register footprint (acc + u [+ q] = 2-3 x the lane's share of the
// row) sets the warp count: f = chunks per lane (H * NCH).
__host__ __device__ constexpr int split_warps(bool cplx, int nch, int var) {
  const int f = (cplx ? 2 : 1) * nch;
  if (var == 0) return f >= 16 ? 13 : 16;                 // 13 x 32 x 128 registers; 8 KB slots
  if (var == 1) return f >= 16 ? 12 : 16;                 // 128 + ~45 registers -> 168 at 12 warps (3 per sub-partition)
  if (var == 2) return f >= 16 ? 8 : (f >= 8 ? 12 : 16);  // 192 + ~45 -> 255 at 8 warps; 96 + 45 -> 168 at 12
  if (var == 3) return f >= 16 ? 12 : 16;                 // warp pairs: 96 + ~45 registers
  return 16;
}
__host__ __device__ constexpr int split_warps_per_row(int var) { return var >= 3 ? 2 : 1; }

// element value and u for one 4-float group (both halves); OP_CDIST runs on packed pairs (FADD2 / FMUL2 / FFMA2)
template <int OP>
__device__ __forceinline__ void unit_group(const float (&q0)[4], const float (&q1)[4], const float (&x0)[4],
                                           const float (&x1)[4], float scale, f2 (&u0)[2], f2 (&u1)[2], float &part,
                                           f2 &part2) {
  if constexpr (OP == OP_CDIST) {
#pragma unroll
    for (int j = 0; j < 4; j += 2) {
      const f2 av = sub2(pack2(q0[j], q0[j + 1]), pack2(x0[j], x0[j + 1]));
      const f2 bv = sub2(pack2(q1[j], q1[j + 1]), pack2(x1[j], x1[j + 1]));
      // |q - x|^2 + FLT_MIN: the guard of the reciprocal square root rides in the FMA chain (it is absorbed by rounding
      // for every |q - x| > 1e-15); at q == x the differences are exactly 0, so u = 0 * finite = 0 (torch's norm subgradient)
      const f2 m2 = fma2(bv, bv, fma2(av, av, pack2(kFltMin, kFltMin)));
      float m2a, m2b;
      unpack2(m2, m2a, m2b);
      const f2 inv = pack2(rsqrt_fast(m2a), rsqrt_fast(m2b));
      u0[j >> 1] = mul2(av, inv);
      u1[j >> 1] = mul2(bv, inv);
      part2 = fma2(m2, inv, part2);                        // += |q - x|
    }
  } else {
    float a0[4], a1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) part += op_unit<OP>(q0[j], q1[j], x0[j], x1[j], scale, a0[j], a1[j]);
    u0[0] = pack2(a0[0], a0[1]); u0[1] = pack2(a0[2], a0[3]);
    u1[0] = pack2(a1[0], a1[1]); u1[1] = pack2(a1[2], a1[3]);
  }
}

template <int MODEL, bool HEAD, int NCH, int VAR>
__global__ void __launch_bounds__(split_warps(op_is_complex(op_of(MODEL, HEAD)), NCH, VAR) * 32, 1)
    row_kernel_split(const RowArgs a, const SplitWs ws) {
  constexpr int OP = op_of(MODEL, HEAD);
  constexpr bool CPLX = op_is_complex(OP);
  constexpr int H = CPLX ? 2 : 1;
  constexpr int V = 4;
  constexpr int DP = 128 * NCH;                 // padded half length (floats)
  constexpr int HS = H * DP;                    // slot size (floats)
  constexpr bool UREG = VAR >= 1, QREG = VAR >= 2;
  constexpr int WPR = split_warps_per_row(VAR);  // warps sharing one candidate row
  constexpr int NCL = NCH / WPR;                 // 128-float chunks (per half) this lane's warp covers
  extern __shared__ __align__(128) float smem[];
  const int Dq4 = (a.De + 3) & ~3;
  const int tid = threadIdx.x, lane = tid & 31;
  // `warp` / `nwarps` index the row groups (one warp, or a pair of warps: hw = which half of the chunks this warp covers)
  const int warp = (tid >> 5) / WPR, nwarps = (blockDim.x >> 5) / WPR, hw = (tid >> 5) % WPR;
  const int c0 = hw * NCL;                        // first chunk of this warp
  // Every row group owns a ring of D = a.ring slots (2..4).  The gather is bound by the bytes in flight per SM against
  // the L2 / DRAM latency (B200, cfg 3: 16 slots of 8 KB per SM gave the same 0.33 ms with 8 warps at 255 registers and
  // with 16 warps at 128; 12 slots were slower), so the ring is as deep as the shared memory allows.
  // layout: [slots: nwarps x D x HS | stage: 2 x (2 De + Dr) | q: HS | dq: De | rot: 2 d | sc[N] | gg[N] | scratch(32) |
  //          stage mbarriers: 2 | ring mbarriers: nwarps x D | pair exchange: nwarps x 4 | parking slot of each group:
  //          nwarps], all derived from `smem`.
  // stage: the head, tail and relation rows of the row's positive triple (the fixed side is one of them), copied by the
  // bulk engine one row AHEAD (double buffer), so that the block-wide phases -- query vector, chain rule, positive
  // triple -- read shared memory instead of waiting on four dependent global-load round trips per row (phase counters
  // r2k: 17 % of the kernel's cycles sat in those two phases).
  const int D = a.ring;
  float *slots = smem + (size_t)(D * warp) * HS;
  const int STG = 2 * a.De + a.Dr;                         // floats per stage buffer (multiple of 4: 16-byte copies)
  float *stage = smem + (size_t)(D * nwarps) * HS;
  float *q = stage + 2 * STG;
  float *dq = q + HS;                           // compact [d | d]
  float *rot = dq + Dq4;                        // [2][d4] cos / sin of the row's relation phases (RotatE)
  const int d4 = (a.d + 3) & ~3;
  float *sc = rot + 2 * d4;                     // [N]
  float *gg = sc + a.N;                         // [N]
  float *scratch = gg + a.N;                    // [32]
  uint64_t *sbars = reinterpret_cast<uint64_t *>(scratch + 32);    // [2] one per stage buffer
  uint64_t *bars = sbars + 2;
  const uint32_t halfbytes = (uint32_t)a.d * 4u;
  uint64_t *gbars = bars + D * warp;                       // this group's mbarriers
  const uint32_t gbars_s = smem_u32(gbars), slots_s = smem_u32(slots);   // (their shared-window addresses)
  uint32_t par = 0;                                         // phase parity of every slot's mbarrier (bit s)
  float *xch = reinterpret_cast<float *>(bars + D * nwarps) + 4 * warp;      // [2 parities][2 halves] partial scores
  int *parks = reinterpret_cast<int *>(reinterpret_cast<float *>(bars + D * nwarps) + 4 * nwarps);

  const float modulus = MODEL == KGE_PROTATE ? __ldg(a.modulus) : 1.f;
  const bool adversarial = a.do_loss && a.loss_kind == KGE_LOSS_NEG_ADVERSARIAL;
  const uint64_t pol_e = l2_policy(a.l2_hints ? 2 : 0);     // entity rows: keep in L2 (see l2_policy)

  {                                                        // zero the pads of every slot and of q (once per CTA)
    const int padn = DP - a.d, nslots = D * nwarps + 1;
    for (int i = tid; i < nslots * H * padn; i += blockDim.x) {
      const int sl = i / (H * padn), r = i % (H * padn);
      float *base = sl < D * nwarps ? smem + (size_t)sl * HS : q;          // (q does not follow the slots directly)
      base[(r / padn) * DP + a.d + (r % padn)] = 0.f;
    }
  }
  if (lane == 0 && hw == 0)
    for (int k = 0; k < D; ++k) mbar_init(gbars + k, 1);
  if (tid == 0) { mbar_init(sbars, 1); mbar_init(sbars + 1, 1); }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();

  // The CTA is persistent (one per SM) and walks its rows; the first D candidates of the NEXT row are issued while the
  // block-wide phases of the current row run (D - 1 right after the candidate loop, the last one as soon as the fold
  // has consumed the accumulators parked in the remaining slot), so every row but the first starts with its bulk
  // copies already in flight.
  int cons = 0;                                            // ring position of the next candidate to consume
  bool primed = false;                                     // the first D candidates of the current row are already issued
  // candidate ids of this warp, 32 at a time (see issue()): the current window, the next window of the same row
  // (fetched 24 candidates ahead) and the first window of the next row (fetched a whole row ahead) -- the id loads
  // never sit in front of a bulk copy (ncu r2d: they did, ~1 us of long-scoreboard stall per 32 candidates and warp).
  // The current window is held clamped as int32 row indices: the single-read path requires nentity < 2^31
  // (split_path_shape_ok), and the row's source address is then one wide multiply-add of the shuffled index.
  int idw = 0;
  int64_t ids_nxt = 0, ids_next_row = 0;
  bool next_row_ready = false;
  int ids_base = -32;
  int cand_rl = 0;
  // (head, relation, tail) of a row, clamped like every gather (the error flag cancels the update)
  auto load_triple = [&](int64_t bb, int64_t &h, int64_t &r, int64_t &t) {
    h = a.positive[bb * 3 + 0]; r = a.positive[bb * 3 + 1]; t = a.positive[bb * 3 + 2];
    if ((uint64_t)h >= (uint64_t)a.nentity || (uint64_t)t >= (uint64_t)a.nentity || (uint64_t)r >= (uint64_t)a.nrelation) {
      if (tid == 0 && a.err) *a.err = 1;
      if ((uint64_t)h >= (uint64_t)a.nentity) h = 0;
      if ((uint64_t)t >= (uint64_t)a.nentity) t = 0;
      if ((uint64_t)r >= (uint64_t)a.nrelation) r = 0;
    }
  };
  auto stage_issue = [&](int buf, int64_t h, int64_t r, int64_t t) {     // thread 0: rows of a triple -> stage[buf]
    float *dst = stage + (size_t)buf * STG;
    const uint32_t eb = (uint32_t)a.De * 4u, rb = (uint32_t)a.Dr * 4u;
    mbar_expect_tx(sbars + buf, 2 * eb + rb);
    bulk_g2s(dst, a.E + h * a.De, eb, sbars + buf);
    bulk_g2s(dst + a.De, a.E + t * a.De, eb, sbars + buf);
    bulk_g2s(dst + 2 * a.De, a.R + r * a.Dr, rb, sbars + buf);
  };
  int64_t hid = 0, rid = 0, tidx = 0, nhid = 0, nrid = 0, ntid = 0;
  if ((int)blockIdx.x < a.row_count) {
    load_triple(a.row_begin + blockIdx.x, hid, rid, tidx);
    if (tid == 0) stage_issue(0, hid, rid, tidx);
  }
  int rowi = 0;                                            // rows done by this CTA: stage buffer = rowi & 1
  for (int rl = blockIdx.x; rl < a.row_count; rl += gridDim.x, ++rowi) {
    const int64_t b = a.row_begin + rl;
    const bool has_next = rl + (int)gridDim.x < a.row_count;
    if (rowi) { hid = nhid; rid = nrid; tidx = ntid; }
    const int64_t fid = HEAD ? tidx : hid;
    const int cb = rowi & 1;
    if (has_next) {                                        // next row's triple: its rows travel under this row's loop
      load_triple(b + gridDim.x, nhid, nrid, ntid);        // (buffer 1 - cb was last read before the previous row's final
      if (tid == 0) stage_issue(cb ^ 1, nhid, nrid, ntid); //  barrier)
    }
    const float *Hs = stage + (size_t)cb * STG, *Ts = Hs + a.De, *Rr = Hs + 2 * a.De;
    const float *F = HEAD ? Ts : Hs;
    const int64_t *cand = a.cand + b * a.cand_stride;
    cand_rl = rl;                                          // row whose candidate list issue() walks
    long long tph = a.phase_cycles ? clock64() : 0;    // debug: cycles per phase of this row (thread 0)

    // candidate ids of this warp (n = warp + j * nwarps), fetched 32 at a time with one load per lane and handed out
    // by shuffle: no dependent global load sits in front of a bulk copy
    // Called by the whole warp (converged).  Per candidate: one shuffle of the window's index and the elected copy issue;
    // the per-id work runs once per window, one candidate per lane.
    auto issue = [&](int s, int j) {                       // j-th candidate of this warp (of the row `cand` points to)
      if (j >= ids_base + 32) {                            // (j is a multiple of 32 here)
        int64_t ids;
        if (j == 0) {
          if (next_row_ready) {
            ids = ids_next_row;
          } else {
            const int n = warp + lane * nwarps;
            ids = n < a.N ? cand[n] : 0;
          }
        } else {
          ids = ids_nxt;
        }
        ids_base = j;
        // the window becomes current: every lane clamps its id once (like every gather), adds it to the histogram of
        // the entity-major pass (one warp-wide reduction for 32 candidates) and keeps an int32 copy on the device --
        // the counting sort reads that instead of the caller's int64 array, which may live in pinned HOST memory
        // (zero-copy batches: this kernel's prefetched window loads are then the only PCIe reads of the ids)
        const int nw = warp + (j + lane) * nwarps;
        if (nw < a.N) {
          if ((uint64_t)ids >= (uint64_t)a.nentity) { if (a.err) *a.err = 1; ids = 0; }
          if (hw == 0) {
            atomicAdd(ws.cnt + ids, 1);
            if (ws.ids32) ws.ids32[(size_t)cand_rl * a.N + nw] = (int)ids;
          }
        }
        idw = (int)ids;
      }
      if (j == ids_base + 8) {                             // next window of this row, 24 candidates ahead of its use
        const int n = warp + (ids_base + 32 + lane) * nwarps;
        ids_nxt = n < a.N ? cand[n] : 0;
      }
      const int id = __shfl_sync(0xffffffffu, idw, j - ids_base);
      if (hw == 0) {
        const float *src = a.E + (size_t)(uint32_t)id * (uint32_t)a.De;
        const uint32_t dst = slots_s + (uint32_t)(s * HS) * 4u;
        bulk_g2s_warp<H, true>(gbars_s + 8u * s, dst, src, dst + DP * 4u, src + a.d, halfbytes, pol_e);
      }
    };
    if (!primed) {
      ids_base = -32;
      for (int k = 0; k < D; ++k)
        if (warp + k * nwarps < a.N) issue((cons + k) % D, k);
    }

    // ---- phase 0: query vector (kept in shared memory and published for the entity-major pass) ----------
    mbar_wait(sbars + cb, (uint32_t)(rowi >> 1) & 1u);    // this row's head / tail / relation rows are in shared memory
    float *qout = ws.Qtab + (size_t)rl * a.De;
    for (int k = tid; k < a.d; k += blockDim.x) {
      if constexpr (MODEL == KGE_ROTATE) {                 // model.py:209-212, once per row
        float sn, cs;
        sincos_rep(fdiv(Rr[k], a.scale), &sn, &cs);
        rot[k] = cs; rot[d4 + k] = sn;
        build_q_rot<HEAD>(F, cs, sn, k, a.d, q, DP);
      } else {
        build_q<MODEL, HEAD>(F, Rr, k, a.d, a.scale, q, DP);
      }
      store_all(a.mir, qout + k, q[k]);                    // (entity-sharded multi-GPU step: every rank gets the row)
      dq[k] = 0.f;
      if (CPLX) { store_all(a.mir, qout + a.d + k, q[DP + k]); dq[a.d + k] = 0.f; }
    }
    __syncthreads();

    if (a.phase_cycles && tid == 0) { const long long t_ = clock64(); atomicAdd(a.phase_cycles + 0, (unsigned long long)(t_ - tph)); tph = t_; }
    // ---- phase 1: per candidate, score (sweep 1) and deferred-normalised dL/dq (sweep 2) ------------------
    f2 acc[NCL][H][2];
#pragma unroll
    for (int i = 0; i < NCL; ++i)
#pragma unroll
      for (int h = 0; h < H; ++h) { acc[i][h][0] = pack2(0.f, 0.f); acc[i][h][1] = pack2(0.f, 0.f); }
    next_row_ready = false;                                // (consumed by the priming above, if it was set)
    if (has_next) {                                        // first id window of the NEXT row: needed after this row's loop
      const int n = warp + lane * nwarps;
      ids_next_row = n < a.N ? (a.cand + (b + gridDim.x) * a.cand_stride)[n] : 0;
    }
    float Mw = -INFINITY;                                  // running max of alpha * s over this warp's rows
    const float *ql = q + c0 * 128 + lane * V;
    float qr[QREG ? NCL : 1][H][V];
    if constexpr (QREG) {
#pragma unroll
      for (int i = 0; i < NCL; ++i) {
        load_shared<V>(qr[i][0], ql + i * 128);
        if constexpr (CPLX) load_shared<V>(qr[i][1], ql + DP + i * 128);
      }
    }
    {
      const bool lead = lane == 0 && hw == 0, timed = a.phase_cycles && tid == 0;
      int it = 0;
      for (int n = warp; n < a.N; n += nwarps, ++it) {
        const int s = cons;
        cons = cons + 1 == D ? 0 : cons + 1;
        { const long long tw_ = timed ? clock64() : 0;
          mbar_wait(gbars_s + 8u * s, (par >> s) & 1u);
          if (timed) atomicAdd(a.phase_cycles + 6, (unsigned long long)(clock64() - tw_)); }
        par ^= 1u << s;
        float *xl = slots + (size_t)s * HS + c0 * 128 + lane * V;
        // sweep 1: element values -> score; u = d(value)/dq stays in registers (VAR >= 1) or is parked in the slot
        float part = 0.f;
        f2 part2 = pack2(0.f, 0.f);
        f2 u[UREG ? NCL : 1][H][2];
        if constexpr (OP == OP_CDIST && QREG) {
          // RotatE, staged so that the MUFU pipe streams: (A) differences and squared moduli of a group of chunks,
          // (B) their reciprocal square roots back to back (the pipe takes a warp instruction every 8 cycles; issued one
          // by one in front of its consumer, each rsqrt exposed its ~20-cycle latency -- ncu r2d: 36 % issue-slot use
          // with no pipe above 40 %), (C) u = (a, b) / |.| and the distance |.| = a u_a + b u_b.
          constexpr int SG = NCL >= 4 ? 4 : NCL;            // chunks per stage group (16 complex dimensions per lane)
          f2 pacc[4] = {pack2(0.f, 0.f), pack2(0.f, 0.f), pack2(0.f, 0.f), pack2(0.f, 0.f)};   // 4 short FFMA2 chains
          const f2 tiny2 = pack2(kFltMin, kFltMin);        // guard of the reciprocal square root, folded into the FMA chain
#pragma unroll
          for (int g0 = 0; g0 < NCL; g0 += SG) {
            f2 m2[SG][2];
#pragma unroll
            for (int i = 0; i < SG; ++i) {
              float x0[V], x1[V];
              load_shared<V>(x0, xl + (g0 + i) * 128);
              load_shared<V>(x1, xl + DP + (g0 + i) * 128);
#pragma unroll
              for (int jj = 0; jj < 2; ++jj) {
                const f2 av = sub2(pack2(qr[g0 + i][0][2 * jj], qr[g0 + i][0][2 * jj + 1]), pack2(x0[2 * jj], x0[2 * jj + 1]));
                const f2 bv = sub2(pack2(qr[g0 + i][1][2 * jj], qr[g0 + i][1][2 * jj + 1]), pack2(x1[2 * jj], x1[2 * jj + 1]));
                u[g0 + i][0][jj] = av;
                u[g0 + i][1][jj] = bv;
                m2[i][jj] = fma2(bv, bv, fma2(av, av, tiny2));
              }
            }
#pragma unroll
            for (int i = 0; i < SG; ++i)
#pragma unroll
              for (int jj = 0; jj < 2; ++jj) {
                float ma, mb;
                unpack2(m2[i][jj], ma, mb);
                // 1/|q - x| (of |q - x|^2 + FLT_MIN, absorbed by rounding for every |q - x| > 1e-15); at q == x the
                // differences are exactly 0, so u = 0 * finite = 0 (torch's norm subgradient)
                m2[i][jj] = pack2(rsqrt_fast(ma), rsqrt_fast(mb));
              }
#pragma unroll
            for (int i = 0; i < SG; ++i)
#pragma unroll
              for (int jj = 0; jj < 2; ++jj) {
                const f2 ua = mul2(u[g0 + i][0][jj], m2[i][jj]);
                pacc[(2 * i + jj) & 1] = fma2(u[g0 + i][0][jj], ua, pacc[(2 * i + jj) & 1]);
                u[g0 + i][0][jj] = ua;
                const f2 ub = mul2(u[g0 + i][1][jj], m2[i][jj]);
                pacc[2 + ((2 * i + jj) & 1)] = fma2(u[g0 + i][1][jj], ub, pacc[2 + ((2 * i + jj) & 1)]);
                u[g0 + i][1][jj] = ub;
              }
            if constexpr (UREG) {
              // (e) this warp's reads of the slot end with the last group's loads (their values fed stage A): hand the
              // slot back to the bulk engine now, ahead of the reduction and the softmax bookkeeping
              if (g0 + SG >= NCL && WPR == 1) {
                __syncwarp();
                if (n + D * nwarps < a.N) issue(s, it + D);
              }
            }
          }
          part2 = add2(add2(pacc[0], pacc[1]), add2(pacc[2], pacc[3]));
        } else
#pragma unroll
        for (int i = 0; i < NCL; ++i) {
          float x0[V], x1[V], q0[V], q1[V];
          load_shared<V>(x0, xl + i * 128);
          if constexpr (CPLX) load_shared<V>(x1, xl + DP + i * 128);
          if constexpr (QREG) {
#pragma unroll
            for (int j = 0; j < V; ++j) { q0[j] = qr[i][0][j]; if constexpr (CPLX) q1[j] = qr[i][1][j]; }
          } else {
            load_shared<V>(q0, ql + i * 128);
            if constexpr (CPLX) load_shared<V>(q1, ql + DP + i * 128);
          }
          if constexpr (!CPLX) {
#pragma unroll
            for (int j = 0; j < V; ++j) { x1[j] = 0.f; q1[j] = 0.f; }
          }
          f2 u0[2], u1[2];
          unit_group<OP>(q0, q1, x0, x1, a.scale, u0, u1, part, part2);
          if constexpr (UREG) {
            u[i][0][0] = u0[0]; u[i][0][1] = u0[1];
            if constexpr (CPLX) { u[i][1][0] = u1[0]; u[i][1][1] = u1[1]; }
          } else if constexpr (!op_unit_is_x(OP)) {
            float t0, t1, t2, t3;
            unpack2(u0[0], t0, t1); unpack2(u0[1], t2, t3);
            *reinterpret_cast<float4 *>(xl + i * 128) = make_float4(t0, t1, t2, t3);
            if constexpr (CPLX) {
              unpack2(u1[0], t0, t1); unpack2(u1[1], t2, t3);
              *reinterpret_cast<float4 *>(xl + DP + i * 128) = make_float4(t0, t1, t2, t3);
            }
          }
        }
        if constexpr (OP == OP_CDIST) {
          float pa, pb;
          unpack2(part2, pa, pb);
          part = pa + pb;
        }
        float coef;
        if constexpr (WPR == 2) {
          // the two halves of the score meet here: one word per warp (double-buffered by candidate parity), one named
          // barrier of the pair; both warps then hold the same sum and run the same softmax bookkeeping
          part = warp_sum(part);
          float *xc = xch + 2 * (it & 1);
          if (lane == 0) xc[hw] = part;
          asm volatile("bar.sync %0, 64;" ::"r"(1 + warp) : "memory");
          part = xc[0] + xc[1];
        }
        if (a.do_loss) {
          if constexpr (WPR == 1) part = warp_sum(part);
          if constexpr (UREG && !(OP == OP_CDIST && QREG && WPR == 1)) {
            // every lane's reads of the slot fed the reduction above: the slot can take the next row already, while
            // the softmax bookkeeping and the accumulate step run from registers
            __syncwarp();
            if (n + D * nwarps < a.N) issue(s, it + D);
          }
          const float sv = finish_score<MODEL>(part, a.gamma, modulus);
          if (lead) sc[n] = sv;                            // (score_out is written from sc after the loop)
          if (adversarial) {                               // online softmax: weight relative to the running max
            const float z = sv * a.alpha;
            if (z > Mw) {
              const float r = expf(Mw - z);                // 0 on the first row (Mw = -inf)
              const f2 r2 = pack2(r, r);
#pragma unroll
              for (int i = 0; i < NCL; ++i)
#pragma unroll
                for (int h = 0; h < H; ++h) { acc[i][h][0] = mul2(acc[i][h][0], r2); acc[i][h][1] = mul2(acc[i][h][1], r2); }
              Mw = z;
            }
            // (2 ulp-level approximations: weights enter dL/dq at 1e-6; the two ex2 are independent MUFU instructions)
            coef = ex2_ftz(kLog2e * (z - Mw)) * sigmoid_fast(sv);
          } else {
            coef = sigmoid_fast(sv);                       // uniform negatives: w = 1/N applied at the end
          }
        } else {
          coef = a.dscore[(int64_t)rl * a.N + n];          // autograd backward: dL/ds is given
          if constexpr (UREG && !(OP == OP_CDIST && QREG && WPR == 1)) {
            __syncwarp();
            if (n + D * nwarps < a.N) issue(s, it + D);
          }
        }
        // sweep 2: acc += coef * u
        const f2 c2 = pack2(coef, coef);
        if constexpr (UREG) {
#pragma unroll
          for (int i = 0; i < NCL; ++i)
#pragma unroll
            for (int h = 0; h < H; ++h) {
              acc[i][h][0] = fma2(c2, u[i][h][0], acc[i][h][0]);
              acc[i][h][1] = fma2(c2, u[i][h][1], acc[i][h][1]);
            }
        } else {
#pragma unroll
          for (int i = 0; i < NCL; ++i) {                  // each lane re-reads exactly the slot words it wrote
            float u0[V], u1[V];
            load_shared<V>(u0, xl + i * 128);
            if constexpr (CPLX) load_shared<V>(u1, xl + DP + i * 128);
            acc[i][0][0] = fma2(c2, pack2(u0[0], u0[1]), acc[i][0][0]);
            acc[i][0][1] = fma2(c2, pack2(u0[2], u0[3]), acc[i][0][1]);
            if constexpr (CPLX) {
              acc[i][1][0] = fma2(c2, pack2(u1[0], u1[1]), acc[i][1][0]);
              acc[i][1][1] = fma2(c2, pack2(u1[2], u1[3]), acc[i][1][1]);
            }
          }
          // the slot was rewritten with generic stores: order them before the bulk engine's next write to it
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (n + D * nwarps < a.N) issue(s, it + D);
        }
      }
    }
    // all issued copies are consumed: the ring is empty at position `cons`.  Next row: candidates 0 .. D-2 go out now,
    // the slot of candidate D-1 parks this row's accumulators for the fold first
    const int ps = (cons + D - 1) % D;
    if (has_next) {
      cand = a.cand + (b + gridDim.x) * a.cand_stride;
      cand_rl = rl + gridDim.x;
      ids_base = -32;
      next_row_ready = true;
      for (int k = 0; k + 1 < D; ++k)
        if (warp + k * nwarps < a.N) issue((cons + k) % D, k);
    }

    if (a.phase_cycles && tid == 0) { const long long t_ = clock64(); atomicAdd(a.phase_cycles + 1, (unsigned long long)(t_ - tph)); tph = t_; }
    // ---- phase 2: loss of this row (model.py:270-288), dL/ds to the workspace ---------------------------------
    float factor;                                           // dL/dq = factor * (folded accumulators)
    if (a.do_loss) {
      __syncthreads();
      const float u = a.weight ? a.weight[b] / a.wsum[0] : a.uniform_u;
      float zmax = 0.f;
      if (adversarial) {
        zmax = -INFINITY;
        for (int n = tid; n < a.N; n += blockDim.x) zmax = fmaxf(zmax, sc[n] * a.alpha);
        zmax = block_reduce(zmax, scratch, true);
      }
      float zsum = 0.f;
      for (int n = tid; n < a.N; n += blockDim.x) {
        const float e = adversarial ? expf(sc[n] * a.alpha - zmax) : 1.f;
        gg[n] = e;
        zsum += e;
      }
      zsum = block_reduce(zsum, scratch, false);
      float lacc = 0.f, gmod = 0.f;
      float *gout = ws.G + (size_t)rl * a.N;
      for (int n = tid; n < a.N; n += blockDim.x) {
        const float w = gg[n] / zsum;
        const float sv = sc[n];
        if (a.score_out) a.score_out[(int64_t)rl * a.N + n] = sv;
        lacc += w * log_sigmoid(-sv);
        const float g = 0.5f * u * w * sigmoid(sv);
        store_all(a.mir, gout + n, g);
        if constexpr (MODEL == KGE_PROTATE) gmod += -g * (a.gamma - sv) / modulus;   // -g * sum|sin|
      }
      const float row_val = block_reduce(lacc, scratch, false);
      if (tid == 0) a.row_loss[b] = row_val;
      if constexpr (MODEL == KGE_PROTATE) {
        gmod = block_reduce(gmod, scratch, false);
        if (tid == 0 && a.gM) red_add1(a.gM, gmod);
      }
      // bring this warp's accumulator to the row's max, then the common scale  (dL/dsum) * u / (2 Z)
      const float r = adversarial ? (Mw == -INFINITY ? 0.f : expf(Mw - zmax)) : 1.f;
      factor = dsum_of<MODEL>(0.5f * u / zsum, modulus) * r;
    } else {
      float *gout = ws.G + (size_t)rl * a.N;
      for (int n = tid; n < a.N; n += blockDim.x) gout[n] = a.dscore[(int64_t)rl * a.N + n];
      if constexpr (MODEL == KGE_PROTATE) {
        // d/dmodulus needs sum|sin| per pair; the backward-only call recomputes it in entity_kernel (rare path)
      }
      factor = dsum_of<MODEL>(1.f, modulus);
      __syncthreads();
    }

    if (a.phase_cycles && tid == 0) { const long long t_ = clock64(); atomicAdd(a.phase_cycles + 2, (unsigned long long)(t_ - tph)); tph = t_; }
    // ---- phase 4: fold the per-warp partial dL/dq.  Each warp parks its (scaled) accumulators in its own idle
    // TMA slot, then every thread sums one k over the warps in fixed order (deterministic, two barriers).
    {
      float *pl = slots + (size_t)ps * HS + c0 * 128 + lane * V;
      if (lane == 0 && hw == 0) parks[warp] = ps;
      const f2 f2v = pack2(factor, factor);
#pragma unroll
      for (int i = 0; i < NCL; ++i) {
#pragma unroll
        for (int h = 0; h < H; ++h) {
          float t0, t1, t2, t3;
          unpack2(mul2(acc[i][h][0], f2v), t0, t1);
          unpack2(mul2(acc[i][h][1], f2v), t2, t3);
          *reinterpret_cast<float4 *>(pl + h * DP + i * 128) = make_float4(t0, t1, t2, t3);
        }
      }
    }
    __syncthreads();
    for (int k = tid; k < a.De; k += blockDim.x) {
      const int kk = (CPLX && k >= a.d) ? DP + (k - a.d) : k;           // compact index -> padded slot offset
      float t = 0.f;
      for (int w = 0; w < nwarps; ++w) t += smem[(size_t)(D * w + parks[w]) * HS + kk];
      dq[k] = t;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // parked / folded slot words vs the next bulk copy
    __syncthreads();
    if (has_next && warp + (D - 1) * nwarps < a.N) issue(ps, D - 1);      // next row, candidate D-1 -> the parking slot
    if (a.phase_cycles && tid == 0) { const long long t_ = clock64(); atomicAdd(a.phase_cycles + 3, (unsigned long long)(t_ - tph)); tph = t_; }
    // ---- phase 5: chain rule into the fixed entity row and the relation row -----------------------------
    // With the fused optimizer (ws.Dvec) the entity-side gradient rows are written to the workspace and reach the
    // entity-major pass as "direct" entries of their target entity; otherwise they are added to gE with atomics.
    // (entity-sharded multi-GPU step: the row goes to the block of the rank that owns the target entity, and only there)
    float *gF = ws.Dvec ? ws.Dvec + (size_t)(3 * rl) * a.De : a.gE + fid * a.De;
    if (a.mir.world > 1) gF = at_rank(a.mir, gF, owner_of(a.mir, fid));
    float *gRr = a.gR + rid * a.Dr;
    for (int k = tid; k < a.d; k += blockDim.x) {
      float dF0, dF1, dR0, dR1;
      if constexpr (MODEL == KGE_ROTATE) chain_q_rot<HEAD>(F, rot[k], rot[d4 + k], dq, k, a.d, a.scale, dF0, dF1, dR0);
      else chain_q<MODEL, HEAD>(F, Rr, dq, k, a.d, a.scale, dF0, dF1, dR0, dR1);
      if (ws.Dvec) {
        gF[k] = dF0;
        if constexpr (CPLX) gF[a.d + k] = dF1;
      } else {
        red_add1(gF + k, dF0);
        if constexpr (CPLX) red_add1(gF + a.d + k, dF1);
      }
      red_add1(gRr + k, dR0);
      if constexpr (MODEL == KGE_COMPLEX) red_add1(gRr + a.d + k, dR1);
    }
    if (a.phase_cycles && tid == 0) { const long long t_ = clock64(); atomicAdd(a.phase_cycles + 4, (unsigned long long)(t_ - tph)); tph = t_; }
    // ---- fused positive triple (model.py:277-279, 'single' mode = the non-head-batch association): the block
    // rebuilds q = fold(h, r), scores the positive tail, and pushes dL/ds+ through the same element functions.
    if (a.pos_row_loss) {
      constexpr int OPS = op_of(MODEL, false);
      __syncthreads();                                      // dq / q of the negatives are no longer needed
      const int64_t ph = hid, pt = tidx;
      if (ws.Dvec && tid < 3) {                             // direct entries of this row: (fixed, head, tail)
        const int64_t target = tid == 0 ? fid : (tid == 1 ? ph : pt);
        store_all(a.mir, ws.dids + 3 * rl + tid, (int)target);
        atomicAdd(ws.cnt + target, 1);
      }
      const float *Hrow = Hs, *Trow = Ts;
      // (tail-batch: q = fold(h, r) is the q of the negatives, still in shared memory)
      if (HEAD) {
        for (int k = tid; k < a.d; k += blockDim.x) {
          if constexpr (MODEL == KGE_ROTATE) build_q_rot<false>(Hrow, rot[k], rot[d4 + k], k, a.d, q, DP);
          else build_q<MODEL, false>(Hrow, Rr, k, a.d, a.scale, q, DP);
        }
        __syncthreads();
      }
      float part = 0.f;
      for (int k = tid; k < a.d; k += blockDim.x)
        part += op_forward<OPS>(q[k], CPLX ? q[DP + k] : 0.f, Trow[k], CPLX ? Trow[a.d + k] : 0.f, a.scale);
      part = block_reduce(part, scratch, false);
      const float sp = finish_score<MODEL>(part, a.gamma, modulus);
      const float up = a.weight ? a.weight[b] / a.wsum[0] : a.uniform_u;
      const float gp = -0.5f * up * sigmoid(-sp);
      if (tid == 0) {
        a.pos_row_loss[b] = log_sigmoid(sp);
        if constexpr (MODEL == KGE_PROTATE) { if (a.gM) red_add1(a.gM, -gp * part); }
      }
      const float gop = dsum_of<MODEL>(gp, modulus);
      float *gT = ws.Dvec ? ws.Dvec + (size_t)(3 * rl + 2) * a.De : a.gE + pt * a.De;
      if (a.mir.world > 1) gT = at_rank(a.mir, gT, owner_of(a.mir, pt));
      for (int k = tid; k < a.d; k += blockDim.x) {
        float dq0 = 0.f, dq1 = 0.f, dx0 = 0.f, dx1 = 0.f;
        op_backward<OPS>(q[k], CPLX ? q[DP + k] : 0.f, Trow[k], CPLX ? Trow[a.d + k] : 0.f, a.scale, gop, dq0, dq1, dx0, dx1);
        dq[k] = dq0;
        if constexpr (CPLX) dq[a.d + k] = dq1;
        if (ws.Dvec) {
          gT[k] = dx0;
          if constexpr (CPLX) gT[a.d + k] = dx1;
        } else {
          red_add1(gT + k, dx0);
          if constexpr (CPLX) red_add1(gT + a.d + k, dx1);
        }
      }
      __syncthreads();
      float *gH = ws.Dvec ? ws.Dvec + (size_t)(3 * rl + 1) * a.De : a.gE + ph * a.De;
      if (a.mir.world > 1) gH = at_rank(a.mir, gH, owner_of(a.mir, ph));
      for (int k = tid; k < a.d; k += blockDim.x) {
        float dF0, dF1, dR0, dR1;
        if constexpr (MODEL == KGE_ROTATE) chain_q_rot<false>(Hrow, rot[k], rot[d4 + k], dq, k, a.d, a.scale, dF0, dF1, dR0);
        else chain_q<MODEL, false>(Hrow, Rr, dq, k, a.d, a.scale, dF0, dF1, dR0, dR1);
        if (ws.Dvec) {
          gH[k] = dF0;
          if constexpr (CPLX) gH[a.d + k] = dF1;
        } else {
          red_add1(gH + k, dF0);
          if constexpr (CPLX) red_add1(gH + a.d + k, dF1);
        }
        red_add1(gRr + k, dR0);
        if constexpr (MODEL == KGE_COMPLEX) red_add1(gRr + a.d + k, dR1);
      }
    }
    if (a.phase_cycles && tid == 0) { const long long t_ = clock64(); atomicAdd(a.phase_cycles + 5, (unsigned long long)(t_ - tph)); tph = t_; }
    __syncthreads();                                        // q / dq / sc are rewritten by the next row
    primed = has_next;
  }
}

// counting sort of the pairs by candidate entity (definitions in kge_train.cu)
__global__ void __launch_bounds__(1024) scan_tiles_kernel(const int *__restrict__ cnt, int *__restrict__ cursor,
                                                          int *__restrict__ tile_tot, int64_t n);
__global__ void __launch_bounds__(1024) scan_apply_kernel(int *__restrict__ cnt, int *__restrict__ cursor,
                                                          const int *__restrict__ tile_tot, int64_t n);
__global__ void scatter_pairs_kernel(const int64_t *__restrict__ cand, int64_t cand_stride, int64_t row_begin, int rows,
                                     int N, int64_t nentity, const int *__restrict__ ids32, const float *__restrict__ G,
                                     const int *__restrict__ dids, int *__restrict__ cursor, int *__restrict__ perm,
                                     float *__restrict__ gsorted);

struct EntArgs {
  float *E;                  // read; written in place by the fused optimizer
  const float *modulus;
  float *gE, *gM;
  const float *gsorted, *Qtab, *Dvec;
  const int *off, *perm;
  int *queue;
  int64_t nentity;
  int64_t ent_begin, ent_count;   // entity range of this launch (slices overlap the NCCL all-reduce in multi-GPU runs)
  int N, d, De;
  int upp;                   // units (float4) per part: ceil(nunits / S)
  int depth;                 // slots per warp in the q-row ring (2..4)
  int l2_hints;              // tag moment traffic evict_first / entity rows evict_last (see l2_policy)
  float scale;
  int need_gmod;             // backward-only pRotatE: accumulate d/dmodulus here
  // fused optimizer (FUSED instantiations)
  float *exp_avg, *exp_avg_sq;
  AdamScalars adam;
  int l3;
  double *reg_partials;      // [gridDim.x]
  const int32_t *err;        // a bad index in this step cancels the update (model.py:86-146 raises before the optimizer)
  Mirror mir;                // entity-sharded multi-GPU step: the updated rows are also stored into every peer's table
};

// One warp per (entity, part) task, S parts per row.  dL/dx is element-wise (no row reduction), so splitting the
// k axis needs no exchange between warps; S = 2 halves the per-thread registers (x and the accumulators) and the
// slot size, which doubles the resident warps (20 per SM; 16 with the fused optimizer, whose epilogue holds a half
// row of both moments next to x and the sums: 128 registers) for latency hiding.
__host__ __device__ constexpr int entity_warps(int parts, bool fused) { return parts == 1 ? 12 : (fused ? 16 : 20); }

__device__ __forceinline__ void prefetch_l2(const void *p, uint32_t bytes, uint64_t pol) {
  asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(p), "r"(bytes), "l"(pol) : "memory");
}

template <int MODEL, bool HEAD, int S, bool FUSED>
__global__ void __launch_bounds__(entity_warps(S, FUSED) * 32, 1) entity_kernel(const EntArgs a) {
  constexpr int OP = op_of(MODEL, HEAD);
  constexpr bool CPLX = op_is_complex(OP);
  constexpr int H = CPLX ? 2 : 1;
  constexpr int V = 4;
  constexpr int CH = (CPLX ? 8 : 16) / S;
  extern __shared__ __align__(128) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  // a slot holds the H halves of a q segment at the compile-time stride HSTR; lanes past the segment (the pad) read
  // whatever an earlier, longer segment left there -- their x registers are 0 and their accumulators are never stored
  constexpr int HSTR = CH * 32 * V;
  constexpr int slot_floats = H * HSTR;
  // per warp a ring of D slots (D = a.depth, 2..4: the bytes in flight per SM are what hides the L2 latency of the q
  // rows -- ncu r2b: 45 % of the instructions of the depth-2 kernel were mbarrier polls); layout
  // [slots: nwarps x D | mbarriers: nwarps x D] (the launcher sizes 16 bytes per slot for the mbarrier)
  const int D = a.depth;
  float *slots = smem + (size_t)(D * warp) * slot_floats;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + (size_t)(D * nwarps) * slot_floats) + D * warp;
  const uint32_t slots_s = smem_u32(slots), bars_s = smem_u32(bars);   // (their shared-window addresses)
  uint32_t par = 0;                                         // phase parity of every slot's mbarrier (bit s)
  const int nunits = a.d / V;
  const float modulus = MODEL == KGE_PROTATE ? __ldg(a.modulus) : 1.f;
  const int64_t ntasks = a.ent_count * S;
  if constexpr (FUSED) {
    if (a.err && *a.err) return;
  }
  // fused optimizer: the moments stream through L2 once per step (evict_first), the entity rows are what the next step's
  // row kernel gathers at random (evict_last)
  const uint64_t pol_mv = l2_policy(a.l2_hints ? 1 : 0), pol_e = l2_policy(a.l2_hints ? 2 : 0);

  for (int i = tid; i < D * nwarps * slot_floats; i += blockDim.x) smem[i] = 0.f;     // finite pads from the start
  if (lane == 0)
    for (int k = 0; k < D; ++k) mbar_init(bars + k, 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();

  float gmod = 0.f;
  double racc = 0.0;
  for (;;) {
    int t = 0;
    if (lane == 0) t = atomicAdd(a.queue, 1);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= ntasks) break;
    const int e = (int)a.ent_begin + t / S, part = t % S;
    const int beg = a.off[e], end = a.off[e + 1];
    const int ubeg = part * a.upp;                          // first unit of this part
    const int ucnt = min(a.upp, nunits - ubeg);             // units in this part
    if (ucnt <= 0) continue;
    if (!FUSED && beg == end) continue;                     // (the fused optimizer also updates untouched entities)
    const uint32_t segbytes = (uint32_t)ucnt * V * 4u;

    // (row index, dL/ds) of the entity's pairs are fetched 32 at a time, one coalesced load per lane, and handed out
    // by shuffle: no dependent global load sits in front of a bulk copy.  Two windows stay live: (prow, pg) holds pairs
    // pbase .. pbase + 31, which the copies are issued from, and (prow0, pg0) the 32 before, which the consumer -- D
    // pairs behind the copies -- may still be reading.
    int prow = 0, prow0 = 0;
    float pg = 0.f, pg0 = 0.f;
    int pbase = beg - 32;                                   // first pair held in (prow, pg)
    auto refill = [&](int i) {
      pbase = i;
      prow0 = prow; pg0 = pg;
      prow = i + lane < end ? a.perm[i + lane] : 0;
      pg = i + lane < end ? a.gsorted[i + lane] : 0.f;
    };
    // called by the whole warp (converged): one shuffle, then the elected copy issue
    auto issue = [&](int s, int i) {
      if (i >= pbase + 32) refill(i);
      const int row = __shfl_sync(0xffffffffu, prow, i - pbase);
      const float *src = (FUSED && row < 0 ? a.Dvec + (size_t)(uint32_t)(-row - 1) * (uint32_t)a.De
                                           : a.Qtab + (size_t)(uint32_t)row * (uint32_t)a.De) + ubeg * V;
      const uint32_t dst = slots_s + (uint32_t)(s * slot_floats) * 4u;
      bulk_g2s_warp<H, false>(bars_s + 8u * s, dst, src, dst + HSTR * 4u, src + a.d, segbytes);
    };
    for (int k = 0; k < D; ++k)
      if (beg + k < end) issue(k, beg + k);
    if constexpr (FUSED) {
      if (lane == 0) {                                      // the moments of this slice are needed at the end of the task
        const size_t mb = (size_t)e * a.De + ubeg * V;
#pragma unroll
        for (int h = 0; h < H; ++h) {
          prefetch_l2(a.exp_avg + mb + (size_t)h * a.d, segbytes, pol_mv);
          prefetch_l2(a.exp_avg_sq + mb + (size_t)h * a.d, segbytes, pol_mv);
        }
      }
    }

    float *xrow = a.E + (size_t)e * a.De + ubeg * V;
    float x0[CH][V], x1[CPLX ? CH : 1][V];
    f2 acc[CH][H][2];
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      const int u = lane + 32 * i;
#pragma unroll
      for (int j = 0; j < V; ++j) { x0[i][j] = 0.f; if constexpr (CPLX) x1[i][j] = 0.f; }
#pragma unroll
      for (int h = 0; h < H; ++h) { acc[i][h][0] = pack2(0.f, 0.f); acc[i][h][1] = pack2(0.f, 0.f); }
      if (u < ucnt) {
        load_global<V>(x0[i], xrow + u * V);
        if constexpr (CPLX) load_global<V>(x1[i], xrow + a.d + u * V);
      }
    }

    const int nact = (ucnt + 31) >> 5;                    // chunks holding at least one unit: the same for every lane
    int s = 0;
    for (int i = beg; i < end; ++i) {
      // (dL/ds, perm entry) of pair i from the window registers; FUSED: perm entry < 0 = direct gradient row
      const bool cur = i >= pbase;
      const int wl = i - pbase + (cur ? 0 : 32);
      const float g = __shfl_sync(0xffffffffu, cur ? pg : pg0, wl);
      const int row = FUSED ? __shfl_sync(0xffffffffu, cur ? prow : prow0, wl) : 0;
      mbar_wait(bars_s + 8u * s, (par >> s) & 1u);
      par ^= 1u << s;
      const float *ql = slots + (size_t)s * slot_floats + lane * V;
      const float go = dsum_of<MODEL>(g, modulus);
      float vsum = 0.f;
      if (FUSED && row < 0) {
        // a gradient row of a positive triple (written by the row kernel): plain sum
#pragma unroll
        for (int c = 0; c < CH; ++c) {
          if (c < nact) {
            float q0[V], q1[V];
            load_shared<V>(q0, ql + c * 128);
            acc[c][0][0] = add2(acc[c][0][0], pack2(q0[0], q0[1]));
            acc[c][0][1] = add2(acc[c][0][1], pack2(q0[2], q0[3]));
            if constexpr (CPLX) {
              load_shared<V>(q1, ql + HSTR + c * 128);
              acc[c][1][0] = add2(acc[c][1][0], pack2(q1[0], q1[1]));
              acc[c][1][1] = add2(acc[c][1][1], pack2(q1[2], q1[3]));
            }
          }
        }
      } else {
#pragma unroll
        for (int c = 0; c < CH; ++c) {
          if (c < nact) {                                   // warp-uniform; no per-lane bounds guard (see HSTR)
            float q0[V], q1[V];
            load_shared<V>(q0, ql + c * 128);
            if constexpr (CPLX) load_shared<V>(q1, ql + HSTR + c * 128);
            if constexpr (OP == OP_CDIST) {
              // RotatE: d|q - x| / dx on packed pairs (FADD2 / FMUL2 / FFMA2): acc -= (q - x) * go / |q - x|,
              // zero at q == x like the scalar form
              const f2 ngo = pack2(-go, -go), tiny2 = pack2(kFltMin, kFltMin);
#pragma unroll
              for (int j = 0; j < V; j += 2) {
                const f2 av = sub2(pack2(q0[j], q0[j + 1]), pack2(x0[c][j], x0[c][j + 1]));
                const f2 bv = sub2(pack2(q1[j], q1[j + 1]), pack2(x1[c][j], x1[c][j + 1]));
                const f2 m2 = fma2(bv, bv, fma2(av, av, tiny2));       // (+ FLT_MIN: the rsqrt guard, see unit_group)
                float m2a, m2b;
                unpack2(m2, m2a, m2b);
                const f2 inv = mul2(pack2(rsqrt_fast(m2a), rsqrt_fast(m2b)), ngo);
                acc[c][0][j >> 1] = fma2(av, inv, acc[c][0][j >> 1]);
                acc[c][1][j >> 1] = fma2(bv, inv, acc[c][1][j >> 1]);
              }
            } else {
              float ex0[V], ex1[V];
#pragma unroll
              for (int j = 0; j < V; ++j) {
                float dq0, dq1;
                ex0[j] = 0.f; ex1[j] = 0.f;
                float xb = 0.f;
                if constexpr (CPLX) xb = x1[c][j];
                const float val = op_backward<OP>(q0[j], CPLX ? q1[j] : 0.f, x0[c][j], xb, a.scale, go, dq0, dq1, ex0[j], ex1[j]);
                if constexpr (MODEL == KGE_PROTATE) vsum += (lane + 32 * c < ucnt) ? val : 0.f;   // pads must not count
              }
              acc[c][0][0] = add2(acc[c][0][0], pack2(ex0[0], ex0[1]));
              acc[c][0][1] = add2(acc[c][0][1], pack2(ex0[2], ex0[3]));
              if constexpr (CPLX) {
                acc[c][1][0] = add2(acc[c][1][0], pack2(ex1[0], ex1[1]));
                acc[c][1][1] = add2(acc[c][1][1], pack2(ex1[2], ex1[3]));
              }
            }
          }
        }
      }
      __syncwarp();
      if (i + D < end) issue(s, i + D);
      s = s + 1 == D ? 0 : s + 1;
      if constexpr (MODEL == KGE_PROTATE) {
        if (a.need_gmod) gmod += -g * warp_sum(vsum);
      }
    }
    if constexpr (FUSED) {
      // torch.optim.Adam on this warp's slice of the entity row, in place: p is in registers (x), g is the sum above
      const size_t base = (size_t)e * a.De + ubeg * V;
      const bool l3 = a.l3 != 0;
#pragma unroll
      for (int h = 0; h < H; ++h) {
        const size_t hb = base + (size_t)h * a.d;
        float mm[CH][V], vv[CH][V];
#pragma unroll
        for (int c = 0; c < CH; ++c) {
          const int u = lane + 32 * c;
          if (u < ucnt) {
            const float4 m4 = ld4_hint(a.exp_avg + hb + u * V, pol_mv), v4 = ld4_hint(a.exp_avg_sq + hb + u * V, pol_mv);
            mm[c][0] = m4.x; mm[c][1] = m4.y; mm[c][2] = m4.z; mm[c][3] = m4.w;
            vv[c][0] = v4.x; vv[c][1] = v4.y; vv[c][2] = v4.z; vv[c][3] = v4.w;
          }
        }
#pragma unroll
        for (int c = 0; c < CH; ++c) {
          const int u = lane + 32 * c;
          if (u < ucnt) {
            const float *px = h == 0 ? x0[c] : x1[CPLX ? c : 0];
            f2 p01 = pack2(px[0], px[1]), p23 = pack2(px[2], px[3]);
            f2 m01 = pack2(mm[c][0], mm[c][1]), m23 = pack2(mm[c][2], mm[c][3]);
            f2 v01 = pack2(vv[c][0], vv[c][1]), v23 = pack2(vv[c][2], vv[c][3]);
            adam_pair_fast(p01, acc[c][h][0], m01, v01, a.adam, l3, racc);
            adam_pair_fast(p23, acc[c][h][1], m23, v23, a.adam, l3, racc);
            float t0, t1, t2, t3;
            unpack2(p01, t0, t1); unpack2(p23, t2, t3);
            // entity-sharded multi-GPU step: owner computes, every replica takes the same bits -- one multicast store
            // through the NVSwitch, or the local store plus one NVLink store per peer
            if (a.mir.mc_delta) {
              multimem_st_v4(reinterpret_cast<float *>(reinterpret_cast<char *>(a.E + hb + u * V) + a.mir.mc_delta),
                             make_float4(t0, t1, t2, t3));
            } else {
              st4_hint(a.E + hb + u * V, make_float4(t0, t1, t2, t3), pol_e);
              for (int r = 0; r < a.mir.world; ++r)
                if (r != a.mir.rank) *reinterpret_cast<float4 *>(at_rank(a.mir, a.E + hb + u * V, r)) = make_float4(t0, t1, t2, t3);
            }
            unpack2(m01, t0, t1); unpack2(m23, t2, t3);
            st4_hint(a.exp_avg + hb + u * V, make_float4(t0, t1, t2, t3), pol_mv);
            unpack2(v01, t0, t1); unpack2(v23, t2, t3);
            st4_hint(a.exp_avg_sq + hb + u * V, make_float4(t0, t1, t2, t3), pol_mv);
          }
        }
      }
    } else {
      // one fire-and-forget 16-byte reduction per float4 of the (half) gradient row: this warp is the only writer of
      // these words in this kernel, so the sum is as deterministic as a store, and no load latency is exposed
      float *grow = a.gE + (size_t)e * a.De + ubeg * V;
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const int u = lane + 32 * c;
        if (u < ucnt) {
#pragma unroll
          for (int h = 0; h < H; ++h) {
            float t0, t1, t2, t3;
            unpack2(acc[c][h][0], t0, t1);
            unpack2(acc[c][h][1], t2, t3);
            red_add4(grow + h * a.d + u * V, t0, t1, t2, t3);
          }
        }
      }
    }
  }
  if constexpr (MODEL == KGE_PROTATE) {
    if (a.need_gmod && lane == 0 && gmod != 0.f && a.gM) red_add1(a.gM, gmod);
  }
  if constexpr (FUSED) {
    if (a.l3 && a.reg_partials) {                           // sum |x|^3 of the pre-update values (model.py:292-295)
      for (int o = 16; o > 0; o >>= 1) racc += __shfl_xor_sync(0xffffffffu, racc, o);
      if (lane == 0) atomicAdd(a.reg_partials + blockIdx.x, racc);
    }
  }
}

}  // namespace kge
