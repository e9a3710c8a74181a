// Renderer backward, default decoder shape (trunk/opacity/colour = 2/2/2 layers, hidden 32, C in {16,32}, <= 3 colours):
// thread-per-sample tcgen05 kernel, see lp_render_tc.cuh for the scheme and DESIGN.md section 4.
//
// Per step and group of 128 rays: forward recompute (three round trips to the tensor core, bf16 hi+lo three-product
// form = fp32-grade), compositing gradient per thread, then the input-gradient chain d_t -> d_h1 -> d_x0.  SURVEY.md H3:
// only the forward / recompute needs fp32-grade products.  The widest input-gradient product, [d_ho | d_hc] (K = 64) ->
// d_t, is ONE kind::tf32 product: the gradient row goes to tensor memory as rounded fp32 words (no hi/lo split, a
// third of the MMAs), its transposed weights are a tf32 K-major tile.  With all three products in TF32 the grid
// gradient measured 0.8-1.0e-3 off the reference's Triton kernels on the same B200 (profiles/gpu_comparator_r2.md) --
// at north_star's 1e-3 bar -- so d_t -> d_h1 -> d_x0 keep the three-product bf16 form.
// The parameter gradients dW = X^T dY are MN-major bf16 tile products accumulated in tensor memory for the whole kernel.
//
// Reference semantics: lightplane/triton_src/templates/renderer_bw.py:89-627.
#pragma once

#include "lp_render_tc.cuh"

namespace lptc {

// tensor-memory columns shared by the CTA: the parameter-gradient accumulators (A1 x DY, A2 x DYL, encoding x S)
constexpr int BT_W = 320, BT_L = 448, BT_ENC = 464;

LP_DEVICE void lp_put_w_tf32(unsigned char* sm, int off, int n, int k, int K, float w) {
  *reinterpret_cast<unsigned*>(sm + off + (n >> 3) * (K >> 2) * 128 + (k >> 2) * 128 + (n & 7) * 16 + (k & 3) * 4) = lp_tf32_rna(w);
}
// store a row of N gradients as this thread's row of a kind::tf32 A operand (one fp32 word per column)
template <int N>
LP_DEVICE void lp_stage_row_tf32(unsigned taddr, const float (&x)[N]) {
  unsigned r[N];
#pragma unroll
  for (int j = 0; j < N; ++j) r[j] = lp_tf32_rna(x[j]);
  lp_tmem_st<N>(taddr, r);
}
// issuer wi of 4: k-steps wi, wi+4, ... of a tf32 product (K = 8 per MMA: 8 A columns, 256 B of the weight tile)
LP_DEVICE void lp_issue_tf32_part(unsigned tbase, int d_col, int a_col, lp_kdesc_t w, int ksteps, int k0, int nstride, int n, int wi) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int ks = wi + 4 * j;
    if (ks < ksteps) lp_tc_mma_ts(true, tbase + d_col, tbase + a_col + 8 * ks, lp_tc_kadv(w, (k0 + ks) * 256), nstride, n, 1);
  }
}

// Precision of the widest input-gradient product [d_ho | d_hc] (K = 64) -> d_t: 0 = three-product bf16 hi+lo form like
// the recompute (grid gradient ~3e-5 off the fp64 oracle), 1 = one kind::tf32 product (a third fewer MMAs, no hi/lo
// split of 64 values per sample; measured -1.5 ms on the headline backward, grid gradient 0.6-0.9e-3 off the oracle
// and the reference's Triton kernels: inside north_star's 1e-3 but without margin, hence not the default).
#ifndef LP_BWD_XT_TF32
#define LP_BWD_XT_TF32 0
#endif
#ifdef LP_ABL_NO_DW
#define LP_ABL_DW(x)
#else
#define LP_ABL_DW(x) x
#endif

// =====================================================================================================================
// Warp-specialised backward: WHO does what
//
//   threads   0..255  two decoder groups (128 threads = 128 rays each): recompute, compositing gradient, input-gradient
//                     chain, parameter-gradient tiles -- everything that talks to the tensor core;
//   threads 256..511  two memory groups, thread i of memory group g serving ray i of decoder group g: sample positions,
//                     the grid gather (-> the first layer's A operand in tensor memory + its dW tile), and the
//                     grid-gradient scatter (the last product's accumulator -> red.global.add.v4).
//
// The memory-bound, long-latency work (L2 gathers, reductions) thereby leaves the decoder threads' instruction streams
// and registers (setmaxnreg: 168 vs 88 registers), runs one step ahead / one step behind them, and the SM holds 16
// instead of 8 warps.  A decoder group never waits for its last product of a step (d_x0 and the dW GEMM are consumed
// by the memory group / the next step): five waited round trips per step instead of six.
// The ray encoding's share of the colour hidden layer, enc x Wc0 + b, is a per-ray constant: it is evaluated once per
// ray tile on the tensor core and kept in shared memory (it replaces the bias add), which frees the tensor-memory
// columns the first layer's operand needs and removes a third of that layer's MMAs.
//
// Hand-offs (mbarriers; "slot" = one iteration of a ray tile: probe, steps 0..tot-1, fold):
//   x0_full  (128 arrivals, memory -> decoder)  slot's operand staged in tensor memory, its flag (+ occupancy) in smem
//   x0_free  (128, decoder -> memory)           every decoder thread has read the slot's flag and seen the first-layer MMAs done
//                                               (a waiter must never fall two phases behind an mbarrier: the producer may
//                                               only advance once ALL consumers have passed the phase, hence 128 arrivals)
//   xt_full  (128, memory -> decoder leaders)   slot's x0 rows written to the dW tile (after the previous dW GEMM)
//   dx_full  (4, tcgen05.commit)                d_x0 of the slot is in tensor memory
//   dx_free  (128, memory -> decoder leaders)   d_x0 read and its accumulator columns cleared
// =====================================================================================================================
template <int C>
struct SImg {
  using I = Img<C>;
  // transposed weights of the input-gradient products:
  static constexpr int XT = (I::FWD_END + 127) / 128 * 128;  // d_t:  tf32 [32 trunk][64: opacity hidden | colour hidden], K-major:
                                                             //       (n, k) at (n/8)*2048 + (k/4)*128 + (n%8)*16 + (k%4)*4
                                                             //       (LP_BWD_XT_TF32 == 0: bf16 hi at XT, lo at XT + 4096, [32][64] K-major)
  static constexpr int XH_HI = XT + 8192;                    // d_h1: bf16 hi / lo [32][32], K-major as the forward tiles
  static constexpr int XH_LO = XH_HI + 2048;
  static constexpr int X0_HI = XH_LO + 2048;                 // d_x0: bf16 hi / lo [C][32]
  static constexpr int X0_LO = X0_HI + C * 64;
  static constexpr int BARS = X0_LO + C * 64;                // 17 mbarriers + TMEM slot + flags (256 B)
  static constexpr int OCC = BARS + 256;                     // [2 groups][128] floats: occupancy of the slot's samples (scaffold)
  static constexpr int GROUPS = OCC + 1024;
  // per-group dW operand tiles, one stack shared by both products:
  //   chunks: ho 0-3 | hc 4-7 | ones 8 | x0 9.. | h1 | trunk      A2 = chunks 0.. (ho, hc, ones), A1 = chunks 8.. (ones, x0, h1, trunk)
  static constexpr int CH_HO = 0, CH_HC = 4, CH_ONES = 8, CH_X0 = 9, CH_H1 = 9 + C / 8, CH_TR = CH_H1 + 4, CH_END = CH_TR + 4;
  static constexpr int STK = 0;
  static constexpr int DY = STK + CH_END * 2048;             // [d_t | d_ho | d_hc | d_h1]
  static constexpr int DYL = DY + 16 * 2048;                 // [dlogit_0..2, g_raw, 0 x 4] (the product's columns 8..15 read what follows: unused)
  static constexpr int ECB = DYL + 2048;                     // float4 [8][128]: enc x Wc0 + b of the tile's rays
  static constexpr int GROUP_BYTES = ECB + 16384;
  // rows of the A1 window
  static constexpr int R_X0 = 8, R_H1 = 8 + C, R_TR = 40 + C;
};
constexpr int ST_A = 0, ST_X = 64, ST_D = 96, ST_GROUP_COLS = 160;  // X: hi 64.., lo 80..; d_x0 lands in D columns 32..

template <int C>
LP_DEVICE void lp_build_simg(unsigned char* sm, const float* __restrict__ P, const LpDecoder& D) {
  using W = SImg<C>;
  const LpLayer &t0 = D.trunk.l[0], &t1 = D.trunk.l[1], &o0 = D.opacity.l[0], &c0 = D.color.l[0];
  const int tid = threadIdx.x, nth = blockDim.x;
  for (int e = tid; e < 32 * 64; e += nth) {  // B[n = trunk feature][k]: k < 32 opacity hidden k, else colour hidden k-32
    const int n = e >> 6, k = e & 63;
    const float w = k < 32 ? P[o0.w_off + n * o0.N + k] : P[c0.w_off + n * c0.N + (k - 32)];
#if LP_BWD_XT_TF32
    lp_put_w_tf32(sm, W::XT, n, k, 64, w);
#else
    lp_put_w(sm, W::XT, W::XT + 4096, n, k, 64, w);
#endif
  }
  for (int e = tid; e < 32 * 32; e += nth) lp_put_w(sm, W::XH_HI, W::XH_LO, e >> 5, e & 31, 32, P[t1.w_off + (e >> 5) * t1.N + (e & 31)]);
  for (int e = tid; e < C * 32; e += nth) lp_put_w(sm, W::X0_HI, W::X0_LO, e >> 5, e & 31, 32, P[t0.w_off + (e >> 5) * t0.N + (e & 31)]);
}
template <int C>
LP_DEVICE void lp_ws_issue_dw_part(unsigned tmem, unsigned char* gs, int wi) {
  using W = SImg<C>;
  const lp_kdesc_t a1 = lp_tc_mndesc_lo(gs + W::STK + W::CH_ONES * 2048), a2 = lp_tc_mndesc_lo(gs + W::STK),
                   dy = lp_tc_mndesc_lo(gs + W::DY), dyl = lp_tc_mndesc_lo(gs + W::DYL);
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int ks = 2 * wi + j;
    lp_tc_mma_ss_mn(tmem + BT_W, lp_tc_kadv(a1, ks * 256), lp_tc_kadv(dy, ks * 256), 2048, 128, 1);
    lp_tc_mma_ss_mn(tmem + BT_L, lp_tc_kadv(a2, ks * 256), lp_tc_kadv(dyl, ks * 256), 2048, 16, 1);
  }
}
template <int C>
LP_DEVICE void lp_ws_issue_encw_part(unsigned tmem, unsigned char* gs, int wi) {
  using W = SImg<C>;
  const lp_kdesc_t a1 = lp_tc_mndesc_lo(gs + W::STK + W::CH_H1 * 2048), dy = lp_tc_mndesc_lo(gs + W::DY + 8 * 2048);
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int ks = 2 * wi + j;
    lp_tc_mma_ss_mn(tmem + BT_ENC, lp_tc_kadv(a1, ks * 256), lp_tc_kadv(dy, ks * 256), 2048, 32, 1);
  }
}

// Code-size switches (headline backward, 16x8 tile walk; profiles/bench_r2_ablation.md):
//   LP_MLP_COMPACT      1: the two trunk layers / the two last gradient layers are run-time loops of one body each and the
//                       compositing gradient has one call site: -2.5 ms (decoder warps were 30 % instruction-fetch stalled)
//   LP_MEM_SINGLE_LOOP  1: one slot loop with single gather / stage / scatter sites in the memory role: +5 ms -- the
//                       compiler's unrolling of the step loop overlaps one slot's scatter with the next slot's gather
// triplane fast path (lp_render_tc.cuh) in the memory role's gather / scatter: off -- its per-axis state costs the 88-register
// memory threads more spills than the shared index arithmetic saves (measured: backward 44.2 -> 45.0 ms with either; all-in-volume 73.6 -> 69.5 ms with the scatter's)
#ifndef LP_BWD_TRI_GATHER
#define LP_BWD_TRI_GATHER false
#endif
#ifndef LP_BWD_TRI_SCATTER
#define LP_BWD_TRI_SCATTER false
#endif
// packed fp32 pairs (lp_platform.cuh), per use.  Measured (backward ms, headline): none 44.09; decoder split only 43.61, bias only 43.71,
// output heads only 43.27, all three 42.64; all three + the memory role's split 47.67
#ifndef LP_BWD_PK_MEM  // the memory role's x0 split stays scalar: packed, its 88-register threads run the whole backward 5 ms slower
#define LP_BWD_PK_MEM false
#endif
#ifndef LP_BWD_PK_SPLIT
#define LP_BWD_PK_SPLIT true
#endif
#ifndef LP_BWD_PK_BIAS
#define LP_BWD_PK_BIAS true
#endif
#ifndef LP_BWD_PK_HEADS
#define LP_BWD_PK_HEADS true
#endif
#ifndef LP_MLP_COMPACT
#define LP_MLP_COMPACT 1
#endif
#ifndef LP_MEM_SINGLE_LOOP
#define LP_MEM_SINGLE_LOOP 0
#endif
// Register split between the roles (setmaxnreg; the two values add up to 256 = 64 K registers / 256 threads per role).
// C = 16: 168 / 88 (splits down to 152 / 104 measure the same); C = 32: the memory threads hold two 32-float rows and spill at
// 88 registers -- 128 / 128 (no re-allocation at all) makes the cfg5 backward 140.0 -> 118.4 ms (152/104: 132.4, 136/120: 120.3);
// giving the memory threads more than the decoder threads loses again (final build: 128/128 110.8 ms, 120/136 115.2, 112/144 117.2).
#ifndef LP_WS_REGS_MEM
#define LP_WS_REGS_MEM(C) ((C) == 16 ? 88 : 128)
#endif
#define LP_WS_REGS_MLP(C) (256 - LP_WS_REGS_MEM(C))
// With ray-geometry gradients (RAYG) the memory threads also hold the ray's six gradient sums and the re-gather's state
#ifndef LP_WS_REGS_MEM_RAYG
#define LP_WS_REGS_MEM_RAYG(C) ((C) == 16 ? 104 : 128)
#endif

// RAYG: also the gradients w.r.t. the rays' origins and directions (io.g_org / io.g_dir, either may be NULL).  Only the
// memory role changes: when it consumes a slot's d_x0 it re-gathers the sample's tap rows and forms
// g_j = sum_t <v_t, d_x0> grad w_t (lp_pos_grad) and J_c^T g_j; the owner thread of a ray sums them over the ray's samples.
template <int C, bool SCAF, bool RAYG>
__global__ void __launch_bounds__(512, 1) lp_render_bwd_ws_kernel(LpRays R, LpMarch M, LpDecoder D, LpGridSet G, LpGridSet SC,
                                                                   const float* __restrict__ params, LpBwdIo io) {
  using I = Img<C>;
  using W = SImg<C>;
  LP_DYN_SMEM(unsigned char, sm);
  // warp index through a broadcast shuffle: the compiler then knows that everything derived from it (group, tensor-memory
  // and shared-memory operand addresses, mbarrier addresses) is warp-uniform and keeps it on the uniform datapath --
  // otherwise every tcgen05.mma / commit / mbarrier operation is wrapped in an elect + R2UR.BROADCAST "waterfall" loop
  const int tid = threadIdx.x, lane = tid & 31, warp = LP_WARP_UNIFORM(tid >> 5);
  const bool is_mlp = warp < 8;
  const int grp = (warp & 7) >> 2, s = tid % GT, wig = warp & 3;
  // mbarriers of group g at bars[8g + ..]: 0 round trips, 1 dW, 2 x0_full, 3 x0_free, 4 xt_full, 5 dx_full, 6 dx_free,
  // 7 first round trip of a slot (no group barrier precedes it, so it must not share a phase sequence with the others); bars[16] init
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(sm + W::BARS);
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 18);
  int* flags = reinterpret_cast<int*>(bars + 20) + 2 * grp;  // [2]: 0 every sample of the slot is empty, 1 full slot, 2 unoccupied (scaffold)
  float* occs = reinterpret_cast<float*>(sm + W::OCC) + grp * GT;
  unsigned char* gs = sm + W::GROUPS + grp * W::GROUP_BYTES;
  lp_build_img<C>(sm, params, D);
  lp_build_simg<C>(sm, params, D);
  for (int e = tid; e < 2 * W::GROUP_BYTES / 16; e += blockDim.x) reinterpret_cast<uint4*>(sm + W::GROUPS)[e] = make_uint4(0u, 0u, 0u, 0u);
  __syncthreads();
  if (is_mlp)  // the row of ones (bf16 1.0): first row of chunk CH_ONES
    *reinterpret_cast<unsigned short*>(gs + W::STK + W::CH_ONES * 2048 + (s >> 3) * 128 + (s & 7) * 16) = 0x3F80;
  if (tid == 0) {
    for (int g = 0; g < 2; ++g) {
      lp_mbar_init(bars + 8 * g + 0, 4); lp_mbar_init(bars + 8 * g + 1, 4); lp_mbar_init(bars + 8 * g + 2, GT);
      lp_mbar_init(bars + 8 * g + 3, GT); lp_mbar_init(bars + 8 * g + 4, GT); lp_mbar_init(bars + 8 * g + 5, 4);
      lp_mbar_init(bars + 8 * g + 6, GT); lp_mbar_init(bars + 8 * g + 7, 4);
    }
    lp_mbar_init(bars + 16, 1);
    lp_mbar_init_fence();
  }
  if (tid < 32) lp_tmem_alloc512(tmem_slot);
  lp_fence_async_smem();
  lp_tc_fence_before();
  __syncthreads();
  lp_tc_fence_after();
  const unsigned tmem = LP_WARP_UNIFORM(*tmem_slot);
  if (tid == 0) {  // zero the dW accumulators: products of the (all-zero) gradient tiles with accumulate off
    const lp_kdesc_t a1 = lp_tc_mndesc_lo(gs + W::STK + W::CH_ONES * 2048), a2 = lp_tc_mndesc_lo(gs + W::STK),
                     dy = lp_tc_mndesc_lo(gs + W::DY), dyl = lp_tc_mndesc_lo(gs + W::DYL), ae = lp_tc_mndesc_lo(gs + W::STK + W::CH_H1 * 2048);
    for (int ks = 0; ks < 8; ++ks) {
      lp_tc_mma_ss_mn(tmem + BT_W, lp_tc_kadv(a1, ks * 256), lp_tc_kadv(dy, ks * 256), 2048, 128, ks > 0);
      lp_tc_mma_ss_mn(tmem + BT_L, lp_tc_kadv(a2, ks * 256), lp_tc_kadv(dyl, ks * 256), 2048, 16, ks > 0);
      lp_tc_mma_ss_mn(tmem + BT_ENC, lp_tc_kadv(ae, ks * 256), lp_tc_kadv(dy, ks * 256), 2048, 32, ks > 0);
    }
    lp_tc_commit(bars + 16);
  }
  lp_mbar_wait(bars + 16, 0);
  lp_tc_fence_after();
  __syncthreads();

  unsigned long long *bar = bars + 8 * grp, *bar_dw = bar + 1, *x0_full = bar + 2, *x0_free = bar + 3, *xt_full = bar + 4,
                     *dx_full = bar + 5, *dx_free = bar + 6, *bar0 = bar + 7;
  const unsigned tbase = tmem + (unsigned)(grp * ST_GROUP_COLS);
  const unsigned tme = lp_taddr(tbase, wig, 0);
  const int num_tiles = (R.n + GT - 1) / GT;
  const int tot = M.S + M.S_inf;
  const int tile0 = blockIdx.x * 2 + grp, tile_stride = gridDim.x * 2;
  constexpr int REGS_MEM = RAYG ? LP_WS_REGS_MEM_RAYG(C) : LP_WS_REGS_MEM(C), REGS_MLP = 256 - REGS_MEM;

  if (!is_mlp) {
    // =================================================================================================================
    // memory group
    // =================================================================================================================
#if LP_MEM_SINGLE_LOOP
    static_assert(!RAYG, "ray-geometry gradients are implemented in the unrolled memory role only");
    if constexpr (REGS_MEM < 128) LP_SETMAXNREG_DEC(REGS_MEM);
    if constexpr (REGS_MEM > 128) LP_SETMAXNREG_INC(REGS_MEM);
    int n_slot = 0, n_dw = 0, n_dx = 0;  // slots staged; dW GEMMs the decoder group has issued; d_x0 rows consumed
    for (int tile = tile0; tile < num_tiles; tile += tile_stride) {
      const Ray1 me = lp_load_ray1(R, lp_tile_ray(M, tile, s), G.g[0].B);
      struct Pos { float x, y, z, oob; };
      Pos prev = {0.f, 0.f, 0.f, 0.f};
      bool pend = false, pend_scatter = false, any_empty = false;  // a full slot whose d_x0 is still to be consumed / scattered
      // One loop over the tile's slots -- probe (n = -1), steps, fold slot (n = tot), flush (n = tot + 1: nothing is
      // published, the last d_x0 is consumed) -- so that the gather, the staging and the scatter exist ONCE in the
      // instruction stream (the kernel is instruction-cache bound otherwise: profiles/ncu_r2c_bwd.md).
#pragma unroll 1
      for (int n = -1; n <= tot + 1; ++n) {
        const bool probe = n < 0, virt = n == tot, flush = n > tot;
        if (virt && !any_empty) continue;
        int flag = 1;
        float occ = 1.f;
        float x0[C];
#pragma unroll
        for (int c = 0; c < C; ++c) x0[c] = 0.f;
        Pos cur = {0.f, 0.f, 0.f, 0.f};
        if (!probe && !virt && !flush) {
          const Sched sc = lp_sched(n, M);
          float depth, delta;
          lp_depth_delta(sc, me.near, me.far, depth, delta);
          cur.x = me.ox + depth * me.dx; cur.y = me.oy + depth * me.dy; cur.z = me.oz + depth * me.dz;
          if (M.contract) lp_contract(cur.x, cur.y, cur.z);
          cur.oob = M.mask_oob ? lp_in_bounds(cur.x, cur.y, cur.z) : 1.f;
          if (SCAF) occ = lp_nearest(SC, me.b, cur.x, cur.y, cur.z);
          if (SCAF && !lp_bar_any(3 + grp, GT, occ != 0.f)) {
            flag = 2;  // nobody's sample is occupied: the slot changes nothing
          } else {
            const bool hit = lp_gather_regs<C, C, LP_BWD_TRI_GATHER>(G, me.b, cur.x, cur.y, cur.z, cur.oob, x0);
            flag = lp_bar_any(3 + grp, GT, hit) ? 1 : 0;
            any_empty |= flag == 0;
          }
        }
        const bool tile_slot = flag == 1 && !probe && !flush;  // this slot ends with a dW GEMM (and produces a d_x0)
        if (!flush) {
          // ---- publish the slot: operand row (full slots) into tensor memory, flag + occupancy into shared memory ----
          if (n_slot > 0) lp_mbar_wait(x0_free, (n_slot - 1) & 1);
          if (flag == 1) {
            lp_tc_fence_after();
            lp_stage_row<C, 16, LP_BWD_PK_MEM>(tme + ST_X, x0);
            lp_tmem_wait_st();
            lp_tc_fence_before();
          }
          if (SCAF) occs[s] = occ;  // (single buffer: the decoder thread reads it before it releases x0_free)
          if (s == 0) flags[n_slot & 1] = flag;
          lp_mbar_arrive(x0_full);
          ++n_slot;
        }
        if (pend && (tile_slot || flush)) {
          // ---- consume the pending d_x0: read it, clear its accumulator columns, release them, scatter ----
          float dxp[C];
          lp_mbar_wait(dx_full, n_dx & 1);
          ++n_dx;
          lp_tc_fence_after();
          lp_tmem_ld<C>(tme + ST_D + 32, dxp);
          lp_tmem_zero<C>(tme + ST_D + 32);
          lp_tmem_wait_st();
          lp_tc_fence_before();
          lp_mbar_arrive(dx_free);
          if (pend_scatter) {  // (warp-uniform) quad-transposed, footprint-merging reduction into the grid gradient
#pragma unroll
            for (int c = 0; c < C; ++c) dxp[c] *= prev.oob;
            lp_splat_quad<C, LP_BWD_TRI_SCATTER>(G, io.g_grid, me.b, prev.x, prev.y, prev.z, me.active && prev.oob != 0.f, dxp);
          }
          pend = false;
        }
        if (tile_slot) {  // the slot's x0 rows go into the dW tile once the previous GEMM is done
          if (n_dw > 0) lp_mbar_wait(bar_dw, (n_dw - 1) & 1);
          ++n_dw;
          lp_tile_row<C>(gs + W::STK, W::CH_X0, s, x0);
          lp_fence_async_smem();
          lp_mbar_arrive(xt_full);
          pend = true;
          pend_scatter = !virt;  // the fold slot's d_x0 is discarded (zero features touch no texel)
          prev = cur;
        }
      }
      ++n_dw;  // the tile's tail: encoding product
    }
#else
    if constexpr (REGS_MEM < 128) LP_SETMAXNREG_DEC(REGS_MEM);
    if constexpr (REGS_MEM > 128) LP_SETMAXNREG_INC(REGS_MEM);
    int n_slot = 0, n_dw = 0, n_dx = 0;  // slots staged; dW GEMMs the decoder group has issued; d_x0 rows consumed
    for (int tile = tile0; tile < num_tiles; tile += tile_stride) {
      const Ray1 me = lp_load_ray1(R, lp_tile_ray(M, tile, s), G.g[0].B);
      struct Pos { float x, y, z, oob, t; };  // t: depth (RAYG)
      Pos prev = {0.f, 0.f, 0.f, 0.f, 0.f};
      bool pend = false, any_empty = false;  // a full slot whose d_x0 is still to be scattered
      float go[3] = {0.f, 0.f, 0.f}, gd[3] = {0.f, 0.f, 0.f};  // RAYG: dL/d origin, dL/d direction of the thread's ray
      // consume the d_x0 of the pending slot: read it, clear its accumulator columns, release them, scatter
      auto drain = [&](bool scatter) {
        float dxp[C];
        lp_mbar_wait(dx_full, n_dx & 1);
        ++n_dx;
        lp_tc_fence_after();
        lp_tmem_ld<C>(tme + ST_D + 32, dxp);
        lp_tmem_zero<C>(tme + ST_D + 32);
        lp_tmem_wait_st();
        lp_tc_fence_before();
        lp_mbar_arrive(dx_free);
        if (scatter) {  // (warp-uniform) quad-transposed, footprint-merging reduction into the grid gradient
#pragma unroll
          for (int c = 0; c < C; ++c) dxp[c] *= prev.oob;
          if constexpr (RAYG) {
            if (prev.oob != 0.f) {  // re-gather the taps (L2-resident), weighted by their weight gradients
              float g[3] = {0.f, 0.f, 0.f};
              lp_pos_grad(G, me.b, prev.x, prev.y, prev.z, [&](const float* row) {
                float acc = 0.f;
#pragma unroll
                for (int k = 0; k < C / 4; ++k) {
                  const float4 v = lp_ldg4(row + 4 * k);
                  acc = fmaf(v.x, dxp[4 * k], acc); acc = fmaf(v.y, dxp[4 * k + 1], acc);
                  acc = fmaf(v.z, dxp[4 * k + 2], acc); acc = fmaf(v.w, dxp[4 * k + 3], acc);
                }
                return acc;
              }, g[0], g[1], g[2]);
              if (M.contract) lp_contract_vjp(me.ox + prev.t * me.dx, me.oy + prev.t * me.dy, me.oz + prev.t * me.dz, g[0], g[1], g[2]);
#pragma unroll
              for (int k = 0; k < 3; ++k) { go[k] += g[k]; gd[k] = fmaf(prev.t, g[k], gd[k]); }
            }
          }
          lp_splat_quad<C, LP_BWD_TRI_SCATTER>(G, io.g_grid, me.b, prev.x, prev.y, prev.z, me.active && prev.oob != 0.f, dxp);
        }
      };
      // publish one slot: operand row (full slots) into tensor memory, flag + occupancy into shared memory
      auto publish = [&](int flag, const float (&x0)[C], float occ, bool tile_too) {
        if (n_slot > 0) lp_mbar_wait(x0_free, (n_slot - 1) & 1);
        if (flag == 1) {
          lp_tc_fence_after();
          lp_stage_row<C, 16, LP_BWD_PK_MEM>(tme + ST_X, x0);
          lp_tmem_wait_st();
          lp_tc_fence_before();
        }
        if (SCAF) occs[s] = occ;  // (single buffer: the decoder thread reads it before it releases x0_free)
        if (s == 0) flags[n_slot & 1] = flag;
        lp_mbar_arrive(x0_full);
        ++n_slot;
        if (flag == 1 && tile_too) {  // this slot ends with a dW GEMM: its x0 rows go into the tile once the previous GEMM is done
          if (pend) { drain(true); pend = false; }
          if (n_dw > 0) lp_mbar_wait(bar_dw, (n_dw - 1) & 1);
          ++n_dw;
          lp_tile_row<C>(gs + W::STK, W::CH_X0, s, x0);
          lp_fence_async_smem();
          lp_mbar_arrive(xt_full);
        }
      };
      {  // probe slot: zero features
        float z0[C];
#pragma unroll
        for (int c = 0; c < C; ++c) z0[c] = 0.f;
        publish(1, z0, 1.f, false);
      }
      for (int step = 0; step < tot; ++step) {
        const Sched sc = lp_sched(step, M);
        float depth, delta;
        lp_depth_delta(sc, me.near, me.far, depth, delta);
        Pos cur;
        cur.x = me.ox + depth * me.dx; cur.y = me.oy + depth * me.dy; cur.z = me.oz + depth * me.dz;
        if constexpr (RAYG) cur.t = depth;
        if (M.contract) lp_contract(cur.x, cur.y, cur.z);
        cur.oob = M.mask_oob ? lp_in_bounds(cur.x, cur.y, cur.z) : 1.f;
        const float occ = SCAF ? lp_nearest(SC, me.b, cur.x, cur.y, cur.z) : 1.f;
        if (SCAF && !lp_bar_any(3 + grp, GT, occ != 0.f)) {  // nobody's sample is occupied: the slot changes nothing
          float z0[C];
#pragma unroll
          for (int c = 0; c < C; ++c) z0[c] = 0.f;
          publish(2, z0, 0.f, false);
          continue;
        }
        float x0[C];
        const bool hit = lp_gather_regs<C, C, LP_BWD_TRI_GATHER>(G, me.b, cur.x, cur.y, cur.z, cur.oob, x0);
        const bool full = lp_bar_any(3 + grp, GT, hit);
        any_empty |= !full;
        publish(full ? 1 : 0, x0, occ, true);
        if (full) { prev = cur; pend = true; }
      }
      if (any_empty) {  // fold slot: zero features, its d_x0 is discarded
        float z0[C];
#pragma unroll
        for (int c = 0; c < C; ++c) z0[c] = 0.f;
        publish(1, z0, 1.f, true);
        drain(false);
      } else if (pend) {
        drain(true);
      }
      if (RAYG && me.active) {  // each ray of the tile belongs to exactly one memory thread: plain stores
        if (io.g_org) { io.g_org[3 * me.ray] = go[0]; io.g_org[3 * me.ray + 1] = go[1]; io.g_org[3 * me.ray + 2] = go[2]; }
        if (io.g_dir) { io.g_dir[3 * me.ray] = gd[0]; io.g_dir[3 * me.ray + 1] = gd[1]; io.g_dir[3 * me.ray + 2] = gd[2]; }
      }
      ++n_dw;  // the tile's tail: encoding product
    }
#endif
  } else {
    // =================================================================================================================
    // decoder group
    // =================================================================================================================
    if constexpr (REGS_MLP > 128) LP_SETMAXNREG_INC(REGS_MLP);
    if constexpr (REGS_MLP < 128) LP_SETMAXNREG_DEC(REGS_MLP);
    // one elected lane (elect.sync) of each of the group's four warps issues its share of every product
    const int wi = wig;
    const float* F = reinterpret_cast<const float*>(sm + I::F32);
    const float4* ecb = reinterpret_cast<const float4*>(gs + W::ECB) + s;
    lp_tmem_zero<32>(tme + ST_D);
    lp_tmem_zero<32>(tme + ST_D + 32);
    const lp_kdesc_t w_t0h = lp_tc_kdesc_lo(sm + I::T0_HI), w_t0l = lp_tc_kdesc_lo(sm + I::T0_LO),
                     w_t1h = lp_tc_kdesc_lo(sm + I::T1_HI), w_t1l = lp_tc_kdesc_lo(sm + I::T1_LO),
                     w_och = lp_tc_kdesc_lo(sm + I::OC_HI), w_ocl = lp_tc_kdesc_lo(sm + I::OC_LO),
                     w_xt = lp_tc_kdesc_lo(sm + W::XT), w_xtl = lp_tc_kdesc_lo(sm + W::XT + 4096), w_xhh = lp_tc_kdesc_lo(sm + W::XH_HI), w_xhl = lp_tc_kdesc_lo(sm + W::XH_LO),
                     w_x0h = lp_tc_kdesc_lo(sm + W::X0_HI), w_x0l = lp_tc_kdesc_lo(sm + W::X0_LO);
    int phase = 0, phase0 = 0, n_dw = 0, n_slot = 0, n_dx = 0, n_xt = 0;
#define LP_ISSUE(A, WH, WL, KS, K0, NS, N, LO, WI) lp_issue_layer_part(tbase, ST_D, A, WH, WL, KS, K0, NS, N, LO, WI)
#define LP_ISSUE_D(DC, A, WH, WL, KS, K0, NS, N, LO, WI) lp_issue_layer_part(tbase, DC, A, WH, WL, KS, K0, NS, N, LO, WI)
#define LP_ISSUE_TF32(DC, A, W_, KS, K0, NS, N) lp_issue_tf32_part(tbase, DC, A, W_, KS, K0, NS, N, wi)
#define LP_TC_HANDOFF(ISSUE) LP_TCG_HANDOFF(1 + grp, GT, lp_elect_one(), ISSUE)
#define LP_TC_WAIT() LP_TCG_WAIT(bar, phase)
#define LP_TC_ROUND(ISSUE) LP_TC_HANDOFF(ISSUE) LP_TC_WAIT()

    for (int tile = tile0; tile < num_tiles; tile += tile_stride) {
      const int ray = lp_tile_ray(M, tile, s);
      const bool active = ray < R.n;
      const int q = active ? ray : R.n - 1;
      const float near = R.near[q], far = R.far[q];
      float v[32];
      {  // enc x Wc0 + b -> shared memory (per-ray constant of the colour hidden layer)
        const float4* e4 = reinterpret_cast<const float4*>(R.enc + (long long)q * H);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float4 t = __ldg(e4 + k);
          v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
        }
        lp_stage_row<32, 32, LP_BWD_PK_SPLIT>(tme + ST_A, v);
        LP_TC_ROUND(if (n_dx > 0) lp_mbar_wait(dx_free, (n_dx - 1) & 1);  // D columns 32.. hold the previous tile's last d_x0
                    LP_ISSUE(ST_A, w_och, w_ocl, 2, 2, 1024, 64, 32, wi); lp_tc_commit(bar));
        lp_tmem_ld<32>(tme + ST_D + 32, v);
        lp_tmem_zero<32>(tme + ST_D + 32);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          const_cast<float4*>(ecb)[k * GT] = make_float4(v[4 * k] + F[I::FB + 96 + 4 * k], v[4 * k + 1] + F[I::FB + 97 + 4 * k],
                                                         v[4 * k + 2] + F[I::FB + 98 + 4 * k], v[4 * k + 3] + F[I::FB + 99 + 4 * k]);
      }
      LpCompBwd cb;  // per-ray constants and running state of the compositing gradient
      cb.init(io, q, active, D.n_feat);
      float S[32];  // sum over steps of the colour-hidden gradient
#pragma unroll
      for (int j = 0; j < 32; ++j) S[j] = 0.f;
      float e_raw = 0.f, e_lg0 = 0.f, e_lg1 = 0.f, e_lg2 = 0.f, G_raw = 0.f, L0 = 0.f, L1 = 0.f, L2 = 0.f;
      bool any_empty = false;

#if LP_MLP_COMPACT
#pragma unroll 1
      for (int step = -1; step <= tot; ++step) {
        const bool probe = step < 0, virt = step == tot;
        if (virt && !any_empty) break;
        // ---- the slot's operand, flag and occupancy from the memory group ----
        lp_mbar_wait(x0_full, n_slot & 1);
        const int flag = flags[n_slot & 1];
        const float occ = SCAF ? occs[s] : 1.f;
        ++n_slot;
        if (flag == 2) {  // unoccupied slot (scaffold): nothing happens
          lp_mbar_arrive(x0_free);
          continue;
        }
        float raw = e_raw, lg0 = e_lg0, lg1 = e_lg1, lg2 = e_lg2;  // flag 0: every sample is empty -> the probe's decoder output
        if (flag == 1) {
          // ------------------------------ forward recompute ------------------------------
          if (lp_elect_one()) {
            lp_tc_fence_after();
            LP_ISSUE(ST_X, w_t0h, w_t0l, C / 16, 0, (C / 8) * 128, 32, 16, wi);
            lp_tc_commit(bar0);
          }
          LP_TCG_WAIT(bar0, phase0);
          lp_mbar_arrive(x0_free);  // the operand columns (and the slot's flag) may be overwritten
          if (n_dw > 0) lp_mbar_wait(bar_dw, (n_dw - 1) & 1);  // the previous dW GEMM has consumed the tiles (long done)
          // the two trunk layers: one body (bias + ReLU + dW tile + hi/lo operand + next product), executed twice
#pragma unroll 1
          for (int l = 0; l < 2; ++l) {
            lp_tmem_ld<32>(tme + ST_D, v);
            lp_tmem_zero<32>(tme + ST_D);
            const float* bl = F + I::FB + 32 * l;
            lp_bias_add<32, LP_BWD_PK_BIAS>(v, bl);  // the ReLU rides on the two conversions below
            lp_tile_row_relu<32>(gs + W::STK, l == 0 ? W::CH_H1 : W::CH_TR, s, v);
            lp_stage_row_relu<32, 32, LP_BWD_PK_SPLIT>(tme + ST_A, v);
            // l == 1: opacity | colour hidden; the product overwrites D columns 32.., where the previous slot's d_x0 may still sit
            LP_TC_HANDOFF(if (l == 1 && n_dx > 0) lp_mbar_wait(dx_free, (n_dx - 1) & 1);
                          LP_ISSUE(ST_A, l == 0 ? w_t1h : w_och, l == 0 ? w_t1l : w_ocl, 2, 0, l == 0 ? 512 : 1024, l == 0 ? 32 : 64, 32, wi);
                          lp_tc_commit(bar));
            LP_TC_WAIT();
          }
          {  // output layer (4 wide) on the CUDA cores, exact fp32; two partial sums per output shorten the FMA chains
            lp_tmem_ld<32>(tme + ST_D, v);
            lp_tmem_zero<32>(tme + ST_D);
            lp_bias_relu<32, LP_BWD_PK_BIAS>(v, F + I::FB + 64);
            raw = lp_head_opacity<LP_BWD_PK_HEADS>(v, F + I::FWO, F[I::FBL + 3]);
            lp_tile_row<32>(gs + W::STK, W::CH_HO, s, v);
            lp_tmem_ld<32>(tme + ST_D + 32, v);
            lp_tmem_zero<32>(tme + ST_D + 32);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float4 eb = ecb[k * GT];  // enc x Wc0 + b (stands in for the bias)
              const float2 lo = lp_add2(lp_f2(v[4 * k], v[4 * k + 1]), lp_f2(eb.x, eb.y)), hi = lp_add2(lp_f2(v[4 * k + 2], v[4 * k + 3]), lp_f2(eb.z, eb.w));
              v[4 * k] = fmaxf(lo.x, 0.f); v[4 * k + 1] = fmaxf(lo.y, 0.f); v[4 * k + 2] = fmaxf(hi.x, 0.f); v[4 * k + 3] = fmaxf(hi.y, 0.f);
            }
            lp_head_colour<LP_BWD_PK_HEADS>(v, F + I::FWC, F + I::FBL, lg0, lg1, lg2);
            lp_tile_row<32>(gs + W::STK, W::CH_HC, s, v);
          }
          if (probe) {  // decoder output at zero features, for the compositing of the empty steps
            e_raw = raw; e_lg0 = lg0; e_lg1 = lg1; e_lg2 = lg2;
            // the next slot's first product is issued without a hand-off: everybody must be done with the accumulators
            lp_tmem_wait_st();
            lp_tc_fence_before();
            lp_bar_sync(1 + grp, GT);
            continue;
          }
        }
        // ------------------------------ compositing gradient (one call site for full and empty slots) ------------------------------
        float g_raw = G_raw, dl0 = L0, dl1 = L1, dl2 = L2;  // fold slot: the summed gradients of the tile's empty steps
        if (!virt) {
          const Sched sc = lp_sched(step, M);
          float depth, delta;
          lp_depth_delta(sc, near, far, depth, delta);
          cb.grad(M, ray, step, step == tot - 1, raw, lg0, lg1, lg2, depth, delta, occ, g_raw, dl0, dl1, dl2);
        }
        if (flag == 0) {  // every sample of the group is empty: gradients summed for the fold slot
          G_raw += g_raw; L0 += dl0; L1 += dl1; L2 += dl2;
          any_empty = true;
          lp_mbar_arrive(x0_free);
          continue;
        }
        lp_tile8(gs + W::DYL, 0, s, dl0, dl1, dl2, g_raw, 0.f, 0.f, 0.f, 0.f);
        // ------------------------------ backward sweep ------------------------------
        lp_head_opacity_bwd<LP_BWD_PK_HEADS>(v, F + I::FWO, g_raw);  // d_ho
        lp_gate_row<32>(v, gs + W::STK, W::CH_HO, s);
#if LP_BWD_XT_TF32
        lp_tile_row<32>(gs + W::DY, 4, s, v);
        lp_stage_row_tf32<32>(tme + ST_A, v);
#else
        lp_tile_stage_row<32, 32>(gs + W::DY, 4, s, tme + ST_A, v);  // [d_ho | d_hc]: packed hi words at columns 0..31, lo at 32..63
#endif
        lp_head_colour_bwd<LP_BWD_PK_HEADS>(v, F + I::FWC, dl0, dl1, dl2);  // d_hc
        lp_gate_row<32>(v, gs + W::STK, W::CH_HC, s);
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const float2 t = lp_add2(lp_f2(S[j], S[j + 1]), lp_f2(v[j], v[j + 1]));
          S[j] = t.x; S[j + 1] = t.y;
        }
#if LP_BWD_XT_TF32
        lp_tile_row<32>(gs + W::DY, 8, s, v);
        lp_stage_row_tf32<32>(tme + ST_A + 32, v);
        LP_TC_ROUND(LP_ISSUE_TF32(ST_D, ST_A, w_xt, 8, 0, 2048, 32); lp_tc_commit(bar));
#else
        lp_tile_stage_row<32, 32>(gs + W::DY, 8, s, tme + ST_A + 16, v);
        LP_TC_ROUND(LP_ISSUE(ST_A, w_xt, w_xtl, 4, 0, 1024, 32, 32, wi); lp_tc_commit(bar));
#endif
        // d_t and d_h1: one body (gate + dW tile + hi/lo operand + next product), executed twice; the second product (d_x0,
        // for the memory group) and the dW GEMM that rides on its hand-off are not waited for
#pragma unroll 1
        for (int l = 0; l < 2; ++l) {
          lp_tmem_ld<32>(tme + ST_D, v);
          lp_tmem_zero<32>(tme + ST_D);
          lp_gate_row<32>(v, gs + W::STK, l == 0 ? W::CH_TR : W::CH_H1, s);
          lp_tile_stage_row<32, 32>(gs + W::DY, l == 0 ? 0 : 12, s, tme + ST_A, v);
          if (l == 0) {
            LP_TC_ROUND(LP_ISSUE(ST_A, w_xhh, w_xhl, 2, 0, 512, 32, 32, wi); lp_tc_commit(bar));
          } else {
            lp_fence_async_smem();  // this step's tile writes -> visible to the tensor core
            LP_TC_HANDOFF(LP_ISSUE_D(ST_D + 32, ST_A, w_x0h, w_x0l, 2, 0, 512, C, 32, wi); lp_tc_commit(dx_full);
                          lp_mbar_wait(xt_full, n_xt & 1); LP_ABL_DW(lp_ws_issue_dw_part<C>(tmem, gs, wi)); lp_tc_commit(bar_dw));
          }
        }
        ++n_dw; ++n_dx; ++n_xt;
      }
#else
      for (int step = -1; step <= tot; ++step) {
        const bool probe = step < 0, virt = step == tot;
        if (virt && !any_empty) break;
        // ---- the slot's operand, flag and occupancy from the memory group ----
        lp_mbar_wait(x0_full, n_slot & 1);
        const int flag = flags[n_slot & 1];
        const float occ = SCAF ? occs[s] : 1.f;
        ++n_slot;
        float depth = 0.f, delta = 0.f;
        if (!probe && !virt) {
          const Sched sc = lp_sched(step, M);
          lp_depth_delta(sc, near, far, depth, delta);
        }
        if (flag != 1) {
          if (flag == 0) {  // every sample of the group is empty: decoder output of the probe, gradients summed for the fold slot
            float g_raw, dl0, dl1, dl2;
            cb.grad(M, ray, step, step == tot - 1, e_raw, e_lg0, e_lg1, e_lg2, depth, delta, occ, g_raw, dl0, dl1, dl2);
            G_raw += g_raw; L0 += dl0; L1 += dl1; L2 += dl2;
            any_empty = true;
          }
          lp_mbar_arrive(x0_free);
          continue;
        }
        // ------------------------------ forward recompute ------------------------------
        if (lp_elect_one()) {
          lp_tc_fence_after();
          LP_ISSUE(ST_X, w_t0h, w_t0l, C / 16, 0, (C / 8) * 128, 32, 16, wi);
          lp_tc_commit(bar0);
        }
        LP_TCG_WAIT(bar0, phase0);
        lp_mbar_arrive(x0_free);  // the operand columns (and the slot's flag) may be overwritten
        if (n_dw > 0) lp_mbar_wait(bar_dw, (n_dw - 1) & 1);  // the previous dW GEMM has consumed the tiles (long done)
        lp_tmem_ld<32>(tme + ST_D, v);
        lp_tmem_zero<32>(tme + ST_D);
        lp_bias_add<32, LP_BWD_PK_BIAS>(v, F + I::FB);
        lp_tile_row_relu<32>(gs + W::STK, W::CH_H1, s, v);
        lp_stage_row_relu<32, 32, LP_BWD_PK_SPLIT>(tme + ST_A, v);
        LP_TC_ROUND(LP_ISSUE(ST_A, w_t1h, w_t1l, 2, 0, 512, 32, 32, wi); lp_tc_commit(bar));
        lp_tmem_ld<32>(tme + ST_D, v);
        lp_tmem_zero<32>(tme + ST_D);
        lp_bias_add<32, LP_BWD_PK_BIAS>(v, F + I::FB + 32);
        lp_tile_row_relu<32>(gs + W::STK, W::CH_TR, s, v);
        lp_stage_row_relu<32, 32, LP_BWD_PK_SPLIT>(tme + ST_A, v);
        // opacity | colour hidden: the product overwrites D columns 32.., where the previous slot's d_x0 may still sit
        LP_TC_HANDOFF(if (n_dx > 0) lp_mbar_wait(dx_free, (n_dx - 1) & 1);
                      LP_ISSUE(ST_A, w_och, w_ocl, 2, 0, 1024, 64, 32, wi); lp_tc_commit(bar));
        LP_TC_WAIT();
        float raw, lg0, lg1, lg2;
        {  // output layer (4 wide) on the CUDA cores, exact fp32; two partial sums per output shorten the FMA chains
          lp_tmem_ld<32>(tme + ST_D, v);
          lp_tmem_zero<32>(tme + ST_D);
          lp_bias_relu<32, LP_BWD_PK_BIAS>(v, F + I::FB + 64);
          raw = lp_head_opacity<LP_BWD_PK_HEADS>(v, F + I::FWO, F[I::FBL + 3]);
          lp_tile_row<32>(gs + W::STK, W::CH_HO, s, v);
          lp_tmem_ld<32>(tme + ST_D + 32, v);
          lp_tmem_zero<32>(tme + ST_D + 32);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float4 eb = ecb[k * GT];  // enc x Wc0 + b (stands in for the bias)
            const float2 lo = lp_add2(lp_f2(v[4 * k], v[4 * k + 1]), lp_f2(eb.x, eb.y)), hi = lp_add2(lp_f2(v[4 * k + 2], v[4 * k + 3]), lp_f2(eb.z, eb.w));
            v[4 * k] = fmaxf(lo.x, 0.f); v[4 * k + 1] = fmaxf(lo.y, 0.f); v[4 * k + 2] = fmaxf(hi.x, 0.f); v[4 * k + 3] = fmaxf(hi.y, 0.f);
          }
          lp_head_colour<LP_BWD_PK_HEADS>(v, F + I::FWC, F + I::FBL, lg0, lg1, lg2);
          lp_tile_row<32>(gs + W::STK, W::CH_HC, s, v);
        }
        if (probe) {  // decoder output at zero features, for the compositing of the empty steps
          e_raw = raw; e_lg0 = lg0; e_lg1 = lg1; e_lg2 = lg2;
          // the next slot's first product is issued without a hand-off: everybody must be done with the accumulators
          lp_tmem_wait_st();
          lp_tc_fence_before();
          lp_bar_sync(1 + grp, GT);
          continue;
        }
        // ------------------------------ compositing gradient ------------------------------
        float g_raw, dl0, dl1, dl2;
        if (!virt) cb.grad(M, ray, step, step == tot - 1, raw, lg0, lg1, lg2, depth, delta, occ, g_raw, dl0, dl1, dl2);
        else { g_raw = G_raw; dl0 = L0; dl1 = L1; dl2 = L2; }  // the summed gradients of the tile's empty steps
        lp_tile8(gs + W::DYL, 0, s, dl0, dl1, dl2, g_raw, 0.f, 0.f, 0.f, 0.f);
        // ------------------------------ backward sweep ------------------------------
        lp_head_opacity_bwd<LP_BWD_PK_HEADS>(v, F + I::FWO, g_raw);  // d_ho
        lp_gate_row<32>(v, gs + W::STK, W::CH_HO, s);
#if LP_BWD_XT_TF32
        lp_tile_row<32>(gs + W::DY, 4, s, v);
        lp_stage_row_tf32<32>(tme + ST_A, v);
#else
        lp_tile_stage_row<32, 32>(gs + W::DY, 4, s, tme + ST_A, v);  // [d_ho | d_hc]: packed hi words at columns 0..31, lo at 32..63
#endif
        lp_head_colour_bwd<LP_BWD_PK_HEADS>(v, F + I::FWC, dl0, dl1, dl2);  // d_hc
        lp_gate_row<32>(v, gs + W::STK, W::CH_HC, s);
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const float2 t = lp_add2(lp_f2(S[j], S[j + 1]), lp_f2(v[j], v[j + 1]));
          S[j] = t.x; S[j + 1] = t.y;
        }
#if LP_BWD_XT_TF32
        lp_tile_row<32>(gs + W::DY, 8, s, v);
        lp_stage_row_tf32<32>(tme + ST_A + 32, v);
        LP_TC_ROUND(LP_ISSUE_TF32(ST_D, ST_A, w_xt, 8, 0, 2048, 32); lp_tc_commit(bar));
#else
        lp_tile_stage_row<32, 32>(gs + W::DY, 8, s, tme + ST_A + 16, v);
        LP_TC_ROUND(LP_ISSUE(ST_A, w_xt, w_xtl, 4, 0, 1024, 32, 32, wi); lp_tc_commit(bar));
#endif
        lp_tmem_ld<32>(tme + ST_D, v);
        lp_tmem_zero<32>(tme + ST_D);
        lp_gate_row<32>(v, gs + W::STK, W::CH_TR, s);  // d_t
        lp_tile_stage_row<32, 32>(gs + W::DY, 0, s, tme + ST_A, v);
        LP_TC_ROUND(LP_ISSUE(ST_A, w_xhh, w_xhl, 2, 0, 512, 32, 32, wi); lp_tc_commit(bar));
        lp_tmem_ld<32>(tme + ST_D, v);
        lp_tmem_zero<32>(tme + ST_D);
        lp_gate_row<32>(v, gs + W::STK, W::CH_H1, s);  // d_h1
        lp_tile_stage_row<32, 32>(gs + W::DY, 12, s, tme + ST_A, v);
        lp_fence_async_smem();  // this step's tile writes -> visible to the tensor core
        // last product of the slot: d_x0 (for the memory group) and the dW GEMM; nobody here waits for them
        LP_TC_HANDOFF(LP_ISSUE_D(ST_D + 32, ST_A, w_x0h, w_x0l, 2, 0, 512, C, 32, wi); lp_tc_commit(dx_full);
                      lp_mbar_wait(xt_full, n_xt & 1); LP_ABL_DW(lp_ws_issue_dw_part<C>(tmem, gs, wi)); lp_tc_commit(bar_dw));
        ++n_dw; ++n_dx; ++n_xt;
      }
#endif
      // ---- per-tile tail: encoding gradient = S Wc0^T, and the encoding's share of dWc0 = enc^T S ----
      if (n_dw > 0) lp_mbar_wait(bar_dw, (n_dw - 1) & 1);
      {
        const float4* e4 = reinterpret_cast<const float4*>(R.enc + (long long)q * H);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float4 t = __ldg(e4 + k);
          v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
        }
        lp_tile_row<32>(gs + W::STK, W::CH_H1, s, v);
        lp_tile_row<32>(gs + W::DY, 8, s, S);
#if LP_BWD_XT_TF32
        lp_stage_row_tf32<32>(tme + ST_A + 32, S);  // K index 32..63 of the d_t weight tile = colour hidden
#else
        lp_stage_row<32, 32, LP_BWD_PK_SPLIT>(tme + ST_A, S);        // issued against k-steps 2, 3 of the tile (K index 32..63 = colour hidden)
#endif
        lp_fence_async_smem();
#if LP_BWD_XT_TF32
        LP_TC_ROUND(LP_ISSUE_TF32(ST_D, ST_A + 32, w_xt, 4, 4, 2048, 32); lp_tc_commit(bar);
#else
        LP_TC_ROUND(LP_ISSUE(ST_A, w_xt, w_xtl, 2, 2, 1024, 32, 32, wi); lp_tc_commit(bar);
#endif
                    lp_ws_issue_encw_part<C>(tmem, gs, wi); lp_tc_commit(bar_dw));
        ++n_dw;
        lp_tmem_ld<32>(tme + ST_D, v);
        lp_tmem_zero<32>(tme + ST_D);
        if (active) {
          float4* ge = reinterpret_cast<float4*>(io.g_enc + (long long)ray * H);
#pragma unroll
          for (int k = 0; k < 8; ++k) ge[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
        }
      }
    }
    if (n_dw > 0) lp_mbar_wait(bar_dw, (n_dw - 1) & 1);
#undef LP_TC_ROUND
#undef LP_TC_HANDOFF
#undef LP_TC_WAIT
#undef LP_ISSUE
#undef LP_ISSUE_TF32
#undef LP_ISSUE_D
  }
  // ---- drain, then the CTA's first four warps read the accumulators (TMEM lane = stack row) ----
  lp_tc_fence_before();
  __syncthreads();
  lp_tc_fence_after();
  if (warp < 4) {
    const LpLayer &t0 = D.trunk.l[0], &t1 = D.trunk.l[1], &o0 = D.opacity.l[0], &o1 = D.opacity.l[1],
                  &c0 = D.color.l[0], &c1 = D.color.l[1];
    float v[32];
    const unsigned tl = lp_taddr(tmem, warp, 0);
    const int r = 32 * warp + lane;  // row of the A1 window: ones 0 | x0 8.. | h1 | trunk
    const int kind = r == 0 ? 0 : (r >= W::R_X0 && r < W::R_X0 + C ? 1 : (r >= W::R_H1 && r < W::R_H1 + 32 ? 2 : (r >= W::R_TR && r < W::R_TR + 32 ? 3 : -1)));
    const int idx = kind == 1 ? r - W::R_X0 : (kind == 2 ? r - W::R_H1 : r - W::R_TR);
#pragma unroll
    for (int blk = 0; blk < 4; ++blk) {  // DY column blocks: d_t | d_ho | d_hc | d_h1
      lp_tmem_ld32u(tl + BT_W + 32 * blk, v);
      const LpLayer& Ly = blk == 0 ? t1 : (blk == 1 ? o0 : (blk == 2 ? c0 : t0));
      const int want = blk == 0 ? 2 : (blk == 3 ? 1 : 3);  // the stack rows whose product with this block is a weight gradient
      if (kind == want)
        for (int n = 0; n < 32; ++n) lp_red_add1(io.g_params + Ly.w_off + idx * Ly.N + n, v[n]);
      else if (kind == 0)
        for (int n = 0; n < 32; ++n) lp_red_add1(io.g_params + Ly.b_off + n, v[n]);
    }
    if (warp == 0) {  // encoding rows x step-summed colour-hidden gradient
      lp_tmem_ld32u(tl + BT_ENC, v);
      for (int n = 0; n < 32; ++n) lp_red_add1(io.g_params + c0.w_off + lane * c0.N + n, v[n]);
    }
    // last layer (A2 x DYL): rows 0..31 opacity hidden, 32..63 colour hidden, 64 ones; columns dlogit_0..2, g_raw
    if (warp < 3) {
      lp_tmem_ld32u(tl + BT_L, v);  // 8 valid columns
      if (warp == 0) {
        lp_red_add1(io.g_params + o1.w_off + lane * o1.N, v[3]);
      } else if (warp == 1) {
        for (int c = 0; c < D.n_feat; ++c) lp_red_add1(io.g_params + c1.w_off + lane * c1.N + c, v[c]);
      } else if (lane == 0) {
        for (int c = 0; c < D.n_feat; ++c) lp_red_add1(io.g_params + c1.b_off + c, v[c]);
        lp_red_add1(io.g_params + o1.b_off, v[3]);
      }
    }
  }
  lp_tc_fence_before();
  __syncthreads();
  if (tid < 32) lp_tmem_dealloc512(tmem);
}

template <int C, bool SCAF, bool RAYG>
static int lp_tc_render_backward_t(cudaStream_t st, const LpRenderArgs& a, const float* params, const LpBwdIo& io) {
  const int groups = 2;
  const int tiles = (a.R.n + GT - 1) / GT;
  int blocks = (tiles + groups - 1) / groups;
  const int max_blocks = lp_tc_num_sms();
  if (blocks > max_blocks) blocks = max_blocks;
  const size_t bytes = SImg<C>::GROUPS + (size_t)groups * SImg<C>::GROUP_BYTES;
  if (LP_TC_SET_SMEM((lp_render_bwd_ws_kernel<C, SCAF, RAYG>), bytes)) return LP_ERR_CUDA;
  LP_LAUNCH((lp_render_bwd_ws_kernel<C, SCAF, RAYG>), dim3(blocks), dim3(2 * groups * GT), bytes, st, a.R, a.M, a.D, a.G, a.SC, params, io);
  return LP_OK;
}
template <bool RAYG>
static int lp_tc_render_backward_r(cudaStream_t st, const LpRenderArgs& a, const float* params, const LpBwdIo& io) {
  if (a.use_scaffold)
    return a.D.C == 16 ? lp_tc_render_backward_t<16, true, RAYG>(st, a, params, io) : lp_tc_render_backward_t<32, true, RAYG>(st, a, params, io);
  return a.D.C == 16 ? lp_tc_render_backward_t<16, false, RAYG>(st, a, params, io) : lp_tc_render_backward_t<32, false, RAYG>(st, a, params, io);
}
// rayg: the launch also writes io.g_org / io.g_dir
static inline int lp_tc_render_backward(cudaStream_t st, const LpRenderArgs& a, const float* params, const LpBwdIo& io, bool rayg) {
  return rayg ? lp_tc_render_backward_r<true>(st, a, params, io) : lp_tc_render_backward_r<false>(st, a, params, io);
}

}  // namespace lptc
