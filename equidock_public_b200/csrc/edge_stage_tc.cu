// Edge stage of IEGMN_Layer.forward (rigid_docking_model.py:204-237, 263-292) on the 5th-gen tensor
// cores (tcgen05 / TMEM), fp32-accurate through a 3-way bf16 split of both operands ("bf16x6":
// a*w ~ a0w0 + a0w1 + a1w0 + a0w2 + a1w1 + a2w0, fp32 accumulation in TMEM; measured error below a
// plain fp32 FMA loop, see scripts/tc_probe.cu).
//
// One persistent CTA per SM, 2 tile groups of 256 threads; each group owns one tile of <=128 edges at a time
// (2 threads per edge row: thread (r, half) <-> columns [32 half, +32) of row r <-> TMEM lane r), the two groups run
// out of phase so one's MMA phases overlap the other's epilogues.  Per tile and group:
//   he rows (cp.async.bulk -> smem staging, prefetched one tile ahead) + 15 RBFs
//     -> [he|rbf] bf16x3 -> TMEM (tcgen05.st)                      A operand of GEMM1 (K=48)
//   GEMM1 (18 tcgen05.mma, B = edge_mlp.0.weight[:, 2dh:] bf16x3 resident in smem)
//     -> + gathered Psrc[src] + Pdst[dst] (cp.async into smem), LeakyReLU, LayerNorm (the two halves of a row
//        combine their statistics through smem) -> bf16x3 -> TMEM
//   GEMM2 and GEMM3 on that one A operand (2 x 24 mma, N=64 halves of the stacked panel [W2 ; W3 W2])
//     -> msg (+bias) -> fp32 tile in smem (mean aggregation at the destination nodes)
//     -> coordinate MLP hidden layer -> LeakyReLU, dot w4 -> phi ; x' = eta x0 + (1-eta) x + mean(x_rel phi) in fp64.
// Per-edge activations never leave the SM; weights are read from HBM/L2 once per CTA.
// The kernel is bound by the dependent chain of a tile group, not by a pipe (profiles/r02_edge_variants.txt): the serial tail of
// a tile is kept short (a tile whose nodes all have 10 in-edges -- a k-NN graph -- needs no row_ptr lookups; the next tile's
// coordinate gathers leave two GEMMs early; the coordinate update runs on threads that do no aggregation) and the fp32
// epilogue arithmetic is written on lane pairs (add / mul / fma.f32x2: the same IEEE results in half the instructions).
#include "tc_common.cuh"
#include "dropout.cuh"

namespace eqd {
#define TC_THREADS 512
__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }
#define TC_MAX_TN 32          // destination nodes per tile (Pdst staging rows)
#define TC_LD 68              // fp32 row stride of the staging / msg tile
#define TC_W_BYTES 67584      // 3 splits x (6144 + 8192 + 8192)
#define TC_W1_SPLIT 6144
#define TC_W23_BASE 18432    // [W2 ; W3 W2] stacked, N = 128
#define TC_W23_SPLIT 16384
#define TC_HE_STAGE_FLOATS (EQD_TM * EQD_EDGE_FEATS + 16)

struct TcWgSmem {                         // per warpgroup
  float stage[EQD_TM * TC_LD];            // gathered Psrc rows, later the fp32 msg tile
  float pdst[2][TC_MAX_TN * TC_LD];       // Pdst rows of the tile's destination nodes (prefetched one tile ahead)
  float he[TC_HE_STAGE_FLOATS];           // raw he rows of the tile (bulk-copied, 16B-aligned chunks)
  double xm[EQD_TM * 3];                  // x_rel per edge (scaled by phi in the coordinate update)
  double xs[EQD_TM * 6];                  // x[src], x[dst] of the tile's edges (prefetched one tile ahead)
  double red[EQD_TM * 4];                 // per-row partial reductions exchanged between the two column halves
  int src[2][EQD_TM];
  int dst[2][EQD_TM];
  int rp[2][TC_MAX_TN + 4];
};

struct TcSmem {
  unsigned char w[TC_W_BYTES];            // bf16x3 weights, canonical K-major no-swizzle UMMA layout
  TcWgSmem wg[2];
  unsigned long long w_bar, mma_bar[2], mma2_bar[2], he_bar[2], a_bar[2];
  unsigned int tmem_base;
};

struct EdgeConsts {                       // per-layer vectors, passed by value (constant bank operands)
  float ln_g[64], ln_b[64], b2[64], b3[64], w4[64];
};

// 512 threads = 2 tile groups x 256; in a group, thread (r = q & 127, half = q >> 7) owns columns
// [32*half, 32*half+32) of edge row r (TMEM lane r): two threads per row keep the per-thread register
// footprint <= 128 so that 16 warps (4 per scheduler) hide each other's latencies.
// DROPOUT (training, dropout.cuh): sites 0 (edge_mlp, c2 = drop.c2) and 1 (coors_mlp, c2 + 1).  Each thread generates the keep
// bits of its 32 columns of a site as ONE 32-bit word right before the epilogue that applies them; mask x scale is applied
// after the LeakyReLU (positively homogeneous: lrelu(m s z) = m s lrelu(z)).  The p = 0 instantiation is the inference kernel.
template <bool DROPOUT>
__global__ void __launch_bounds__(TC_THREADS, 1)
edge_stage_tc_kernel(eqd_graph g, eqd_layer_params p, const __grid_constant__ EdgeConsts cst,
                     const float* __restrict__ proj, const double* __restrict__ x_in, const double* __restrict__ x_orig,
                     float* __restrict__ aggr, double* __restrict__ x_out, int* __restrict__ status, int tn, DropoutArgs drop) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  TcSmem& S = *reinterpret_cast<TcSmem*>(smem_raw);
  const int tid = threadIdx.x, wg = tid >> 8, q = tid & 255, half = q >> 7, r = q & 127, warp = tid >> 5;
  TcWgSmem& W = S.wg[wg];
  const int pw = 128 + 3 * p.dhp;
  const int ntiles = (g.n_nodes + tn - 1) / tn;
  const float slope = p.leaky_slope;

  TRACE_START(0);
  // ---- one-time setup: TMEM, barriers, weights (one TMA bulk copy) -------------------------------
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    mbar_init(&S.w_bar, 1);
    mbar_init(&S.mma_bar[0], 1);
    mbar_init(&S.mma_bar[1], 1);
    mbar_init(&S.he_bar[0], 1);
    mbar_init(&S.he_bar[1], 1);
    for (int a = 0; a < 2; ++a) {
      mbar_init(&S.mma2_bar[a], 1);
      mbar_init(&S.a_bar[a], 8);      // one arrival per warp of the tile group: "my part of the A operand is in TMEM"
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(&S.w_bar, TC_W_BYTES);
    bulk_g2s(S.w, p.w_edge_tc, TC_W_BYTES, &S.w_bar);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // warp-uniform copies for the MMA issue path: operands the compiler can prove uniform go straight to uniform
  // registers (UTCHMMA takes UR operands); anything else costs a per-MMA waterfall loop (ELECT / R2UR / BRA.U.ANY)
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int wg_u = warp_u >> 3;
  const bool issuer_warp = (warp_u & 7) == 0;
  const unsigned tmem_base_u = __shfl_sync(0xffffffffu, S.tmem_base, 0);
  const unsigned tmem_wg = tmem_base_u + (unsigned)wg_u * 256;                   // lane 0 (MMA issuer's view)
  const unsigned tmem = tmem_wg + ((unsigned)((warp & 3) * 32) << 16);           // my lane quarter
  const unsigned d_col = tmem + half * 32;                                         // my half of D (64 columns)
  const unsigned a_col = tmem + 128;                                               // A: 3 splits x 32 columns (D: 0..127)
  if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, 0, 1);
  mbar_wait(&S.w_bar, 0);
  unsigned mma_phase = 0, mma2_phase = 0, he_phase = 0, a_phase = 0;
  const unsigned w_saddr = smem_u32(S.w);

  // Prefetch of a tile's indices, Pdst rows and he rows.
  auto prefetch = [&](int tile, int buf, int& e0_out, int& ne_out, int& off_l, int& n_l, int& off_r) {
    const int n0 = tile * tn, nn = min(tn, g.n_nodes - n0);
    const int e0 = __ldg(g.row_ptr + n0), e1 = __ldg(g.row_ptr + n0 + nn);
    const int ne = e1 - e0;
    e0_out = e0;
    ne_out = ne;
    off_l = off_r = 0;
    n_l = 0;
    if (ne <= EQD_TM) {
      if (r < ne) {   // every thread fetches the index its own prefetch_x() reads (no barrier in between)
        if (half == 0) cp_async4(&W.src[buf][r], g.col_src + e0 + r);
        else cp_async4(&W.dst[buf][r], g.edge_dst + e0 + r);
      }
      if (half == 0 && r <= nn) cp_async4(&W.rp[buf][r], g.row_ptr + n0 + r);
      // he rows: [e0, e1) split at the ligand/receptor array boundary; 16-byte aligned bulk copies
      const int el0 = min(e0, g.n_lig_edges), el1 = min(e1, g.n_lig_edges);
      n_l = el1 - el0;
      long sl = 0, sr = 0;
      unsigned bl = 0, br = 0;
      if (n_l > 0) {
        long b0 = (long)el0 * (EQD_EDGE_FEATS * 4), b1 = (long)el1 * (EQD_EDGE_FEATS * 4);
        sl = b0 & ~15L;
        bl = (unsigned)(((b1 + 15) & ~15L) - sl);
        off_l = (int)((b0 - sl) >> 2);
      }
      const int nr = ne - n_l;
      const unsigned dst_r_off = bl;  // receptor part lands after the ligand part (bl is a multiple of 16)
      if (nr > 0) {
        long b0 = (long)(e0 + n_l - g.n_lig_edges) * (EQD_EDGE_FEATS * 4), b1 = (long)(e1 - g.n_lig_edges) * (EQD_EDGE_FEATS * 4);
        sr = b0 & ~15L;
        br = (unsigned)(((b1 + 15) & ~15L) - sr);
        off_r = (int)(dst_r_off >> 2) + (int)((b0 - sr) >> 2);
      }
      for (int idx = q; idx < nn * 16; idx += 256) {   // Pdst rows of the tile's (contiguous) destination nodes
        int row = idx >> 4, c4 = idx & 15;
        cp_async16(&W.pdst[buf][row * TC_LD + c4 * 4], proj + (long)(n0 + row) * pw + 64 + c4 * 4, true);
      }
      if (q == 0) {
        mbar_expect_tx(&S.he_bar[wg], bl + br);
        if (bl) bulk_g2s(W.he, reinterpret_cast<const unsigned char*>(g.he_lig) + sl, bl, &S.he_bar[wg]);
        if (br) bulk_g2s(reinterpret_cast<unsigned char*>(W.he) + dst_r_off, reinterpret_cast<const unsigned char*>(g.he_rec) + sr, br,
                         &S.he_bar[wg]);
      }
    }
    cp_async_commit();
  };
  // Coordinates of a tile's edge endpoints -> smem (needs that tile's indices to have landed).
  auto prefetch_x = [&](int b, int ne_t) {
    if (r < ne_t && ne_t <= EQD_TM) {
      const double* xp = x_in + (long)(half == 0 ? W.src[b][r] : W.dst[b][r]) * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) cp_async8(&W.xs[r * 6 + half * 3 + c], xp + c);
    }
    cp_async_commit();
  };

  int tile = blockIdx.x * 2 + wg;
  const int tstride = gridDim.x * 2;
  const int lane = tid & 31, wrow0 = 32 * (warp & 3);
  const int pair_id = 3 + wg * 4 + (warp & 3);   // named barrier of the two warps that hold rows [wrow0, wrow0 + 32)
  int buf = 0;
  int e0 = 0, ne = 0, off_l = 0, n_l = 0, off_r = 0;
  if (tile < ntiles) {
    prefetch(tile, buf, e0, ne, off_l, n_l, off_r);
    cp_async_wait<0>();
    wg_barrier(wg);
    prefetch_x(buf, ne);
  }

  for (; tile < ntiles; tile += tstride) {
    const int n0 = tile * tn, nn = min(tn, g.n_nodes - n0);
    const bool has_next = tile + tstride < ntiles;
    int e0n = 0, nen = 0, off_ln = 0, n_ln = 0, off_rn = 0;
    if (ne > EQD_TM) {  // in-degree bound violated: flag, skip (uniform per tile group)
      if (q == 0) atomicOr(status + g.n_pairs, EQD_STATUS_DEGREE_OVERFLOW);
      cp_async_wait<0>();
      wg_barrier(wg);
      if (has_next) {
        prefetch(tile + tstride, buf ^ 1, e0n, nen, off_ln, n_ln, off_rn);
        cp_async_wait<0>();
        wg_barrier(wg);
        prefetch_x(buf ^ 1, nen);
      }
      e0 = e0n; ne = nen; off_l = off_ln; n_l = n_ln; off_r = off_rn; buf ^= 1;
      continue;
    }
    // ---- S0/S1: indices + coordinates ready; geometry; [he|rbf] -> TMEM ---------------------------------------
    // Synchronisation inside a tile: two full group barriers (here and before the aggregation).  Everything else is
    // point to point -- each warp announces its part of an A operand on an mbarrier that only the MMA-issuing warp
    // waits for, every warp gathers exactly the Psrc rows it will read itself (warp-local visibility), and the two
    // column halves of a row exchange their LayerNorm statistics through a 64-thread named barrier.
    if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 2);
    cp_async_wait<0>();
    wg_barrier(wg);
    if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 3);
    const bool valid = r < ne;
    const int dn = valid ? W.dst[buf][r] : 0;
    {
      float a1v[24];  // half 0: he[0..23];  half 1: he[24..26], 15 RBFs, 6 zeros
      mbar_wait(&S.he_bar[wg], he_phase);
      he_phase ^= 1;
      if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 4);
      const float* hrow = W.he + (r < n_l ? off_l + r * EQD_EDGE_FEATS : off_r + (r - n_l) * EQD_EDGE_FEATS);
      if (half == 0) {
#pragma unroll
        for (int k = 0; k < 24; ++k) a1v[k] = valid ? hrow[k] : 0.f;
      } else {
        double rx = 0.0, ry = 0.0, rz = 0.0;
        if (valid) {  // u_sub_v :204-205
          rx = W.xs[r * 6 + 0] - W.xs[r * 6 + 3];
          ry = W.xs[r * 6 + 1] - W.xs[r * 6 + 4];
          rz = W.xs[r * 6 + 2] - W.xs[r * 6 + 5];
          W.xm[r * 3 + 0] = rx;
          W.xm[r * 3 + 1] = ry;
          W.xm[r * 3 + 2] = rz;
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) a1v[k] = valid ? hrow[24 + k] : 0.f;
        const float nd2 = valid ? -(float)(rx * rx + ry * ry + rz * rz) : -INFINITY;  // :208-209; padding rows: exp2(-inf) = 0
        // exp(-d^2 / 1.5^q) :210 as ex2.approx(-d^2 * log2(e)/1.5^q): 2 instructions per RBF instead of ~20; the
        // features are <= 1 and the absolute error (<= 2e-7: 2^-22 of ex2 + the rounded scale factor) is below the
        // bf16x3 operand resolution of the GEMM they feed
        constexpr double kS[EQD_N_RBF] = {1.0, 1.5, 2.25, 3.375, 5.0625, 7.59375, 11.390625, 17.0859375, 25.62890625,
                                          38.443359375, 57.6650390625, 86.49755859375, 129.746337890625,
                                          194.6195068359375, 291.92926025390625};
#pragma unroll
        for (int j = 0; j < EQD_N_RBF; ++j)
          a1v[3 + j] = exp2f(nd2 * (float)(1.4426950408889634 / kS[j]));
#pragma unroll
        for (int k = 18; k < 24; ++k) a1v[k] = 0.f;
      }
      unsigned p0[12], p1[12], p2[12];
#pragma unroll
      for (int c = 0; c < 12; ++c) split3_pair(a1v[2 * c], a1v[2 * c + 1], p0[c], p1[c], p2[c]);
      const unsigned ab = a_col + half * 12;
      tmem_st8(ab, p0);      tmem_st4(ab + 8, p0 + 8);
      tmem_st8(ab + 32, p1); tmem_st4(ab + 40, p1 + 8);
      tmem_st8(ab + 64, p2); tmem_st4(ab + 72, p2 + 8);
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&S.a_bar[wg]);
    // ---- GEMM1: [he|rbf] (K=48) x W1e ---------------------------------------------------------------
    if (issuer_warp) {
      if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 5);
      mbar_wait(&S.a_bar[wg_u], a_phase);   // all 8 warps' A columns are in TMEM (and they are done with the he staging)
      a_phase ^= 1;
      if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 6);
      tc_fence_after();
      if (elect_one()) {
        issue_gemm(tmem_wg, tmem_wg + 128, 32, w_saddr, TC_W1_SPLIT, 3);
        umma_commit(&S.mma_bar[wg_u]);
      }
      __syncwarp();
    }
    // Psrc[src] of MY warp's 32 rows x MY column half -> smem (8 lanes per row: 128 contiguous bytes), behind GEMM1
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int grow = wrow0 + i * 4 + (lane >> 3);
      const bool ok = grow < ne;
      const int s_row = ok ? W.src[buf][grow] : 0;
      cp_async16(&W.stage[grow * TC_LD + half * 32 + (lane & 7) * 4], proj + (long)s_row * pw + half * 32 + (lane & 7) * 4, ok);
    }
    cp_async_commit();
    // he staging and the other index / Pdst buffers are free now: prefetch the next tile behind the MMAs
    if (has_next) prefetch(tile + tstride, buf ^ 1, e0n, nen, off_ln, n_ln, off_rn);
    if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 7);
    mbar_wait(&S.mma_bar[wg], mma_phase);
    mma_phase ^= 1;
    tc_fence_after();
    if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 8);
    // ---- epilogue 1: + Psrc[src] + Pdst[dst], LeakyReLU, LayerNorm -> bf16x3 -> TMEM ----------------
    {
      float v[32];
      tmem_ld32f(d_col, v);
      if (has_next) cp_async_wait<1>(); else cp_async_wait<0>();  // my gathers landed (the newest group is the prefetch)
      __syncwarp();                                                  // ... and so did the rest of my warp's
      const int dloc = valid ? dn - n0 : 0;
      const float4* ps = reinterpret_cast<const float4*>(&W.stage[r * TC_LD + half * 32]);
      const float4* pd = reinterpret_cast<const float4*>(&W.pdst[buf][dloc * TC_LD + half * 32]);
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
      {   // The fp32 epilogue arithmetic is written on lane PAIRS (add.f32x2 / mul.f32x2 / fma.f32x2 of sm_100: one instruction,
          // two IEEE results -- bitwise the scalar sequence, ~5 % fewer instructions in this latency-bound kernel)
        float2 s01 = f2(0.f, 0.f), s23 = f2(0.f, 0.f);
        const float2 sl2 = f2(slope, slope);
        unsigned keep = 0;
        if (DROPOUT) keep = dropout_keep32(drop, dropout_key(drop), 8 * half, (unsigned)(e0 + r), drop.c2);
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          float4 a = ps[c4], b = pd[c4];
          float2 x01 = __fadd2_rn(__fadd2_rn(f2(v[c4 * 4 + 0], v[c4 * 4 + 1]), f2(a.x, a.y)), f2(b.x, b.y));
          float2 x23 = __fadd2_rn(__fadd2_rn(f2(v[c4 * 4 + 2], v[c4 * 4 + 3]), f2(a.z, a.w)), f2(b.z, b.w));
          float2 y01 = __fmul2_rn(x01, sl2), y23 = __fmul2_rn(x23, sl2);
          float2 t01 = f2(fmaxf(x01.x, y01.x), fmaxf(x01.y, y01.y)), t23 = f2(fmaxf(x23.x, y23.x), fmaxf(x23.y, y23.y));
          if (DROPOUT) {   // site 0: before the LayerNorm statistics
            t01 = __fmul2_rn(t01, f2(dropout_mul(keep, c4 * 4 + 0, drop.scale), dropout_mul(keep, c4 * 4 + 1, drop.scale)));
            t23 = __fmul2_rn(t23, f2(dropout_mul(keep, c4 * 4 + 2, drop.scale), dropout_mul(keep, c4 * 4 + 3, drop.scale)));
          }
          v[c4 * 4 + 0] = t01.x; v[c4 * 4 + 1] = t01.y; v[c4 * 4 + 2] = t23.x; v[c4 * 4 + 3] = t23.y;
          s01 = __fadd2_rn(s01, t01);
          s23 = __fadd2_rn(s23, t23);
        }
        s4[0] = s01.x; s4[1] = s01.y; s4[2] = s23.x; s4[3] = s23.y;
      }
      // LayerNorm statistics: two-pass over this half (mean_h, M2_h), then the exact pairwise combination
      //   mean = (m0+m1)/2,  M2 = M2_0 + M2_1 + (m0-m1)^2 * 16      (Chan et al.)
      const float mh = ((s4[0] + s4[1]) + (s4[2] + s4[3])) * (1.f / 32.f);
      float q4[4] = {0.f, 0.f, 0.f, 0.f};
      {
        float2 q01 = f2(0.f, 0.f), q23 = f2(0.f, 0.f);
        const float2 nmh = f2(-mh, -mh);
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          float2 d01 = __fadd2_rn(f2(v[c], v[c + 1]), nmh), d23 = __fadd2_rn(f2(v[c + 2], v[c + 3]), nmh);
          q01 = __ffma2_rn(d01, d01, q01);
          q23 = __ffma2_rn(d23, d23, q23);
        }
        q4[0] = q01.x; q4[1] = q01.y; q4[2] = q23.x; q4[3] = q23.y;
      }
      float* redf = reinterpret_cast<float*>(W.red);
      redf[(r * 2 + half) * 2 + 0] = mh;
      redf[(r * 2 + half) * 2 + 1] = (q4[0] + q4[1]) + (q4[2] + q4[3]);
      if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 9);
      pair_barrier(pair_id);   // only the warp that owns the other half of these 32 rows
      const float m0 = redf[r * 4 + 0], m1 = redf[r * 4 + 2];
      const float mean = 0.5f * (m0 + m1);
      const float dm = m0 - m1;
      const float var = (redf[r * 4 + 1] + redf[r * 4 + 3] + dm * dm * 16.f) * (1.f / 64.f);
      const float rstd = 1.f / sqrtf(var + 1e-5f);
      {
        const float2 nm = f2(-mean, -mean), rs2 = f2(rstd, rstd);
#pragma unroll
        for (int c = 0; c < 32; c += 2) {
          float2 t = __fmul2_rn(__fadd2_rn(f2(v[c], v[c + 1]), nm), rs2);
          t = __ffma2_rn(t, f2(cst.ln_g[half * 32 + c], cst.ln_g[half * 32 + c + 1]), f2(cst.ln_b[half * 32 + c], cst.ln_b[half * 32 + c + 1]));
          v[c] = t.x; v[c + 1] = t.y;
        }
      }
      store_half_split3(a_col + half * 16, v);
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&S.a_bar[wg]);
    if (has_next) {
      // The next tile's x[src] / x[dst] gathers go out here, two GEMMs before they are needed (issued in the tail of the tile
      // their latency sat in front of the next tile's first barrier).  xs of this tile was consumed in S0 by the half-1 thread of my row, which has since met me at the LayerNorm pair
      // barrier; my own index of the next tile (fetched behind GEMM1) has landed once my copy groups drain
      cp_async_wait<0>();
      prefetch_x(buf ^ 1, nen);
    }
    // ---- GEMM2 and GEMM3 on the same A operand ------------------------------------------------------------------
    // msg = W2 a1 + b2 (edge_mlp.4) and the coordinate MLP's hidden pre-activation W3 msg + b3 =
    // (W3 W2) a1 + (W3 b2 + b3) are both linear in a1: the stacked panel [W2 ; W3 W2] gives them from one A operand
    // (no bf16x3 split of msg, no second TMEM store).  Issued as two N=64 halves with their own completion barriers so
    // that the msg epilogue runs under the second half's MMAs.
    if (issuer_warp) {
      if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 10);
      mbar_wait(&S.a_bar[wg_u], a_phase);
      a_phase ^= 1;
      tc_fence_after();
      if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 11);
      if (elect_one()) {
        const int pa[6] = {2, 0, 1, 1, 0, 0}, pb[6] = {0, 2, 1, 0, 1, 0};
#pragma unroll
        for (int hn = 0; hn < 2; ++hn) {
          unsigned accum = 0;
#pragma unroll
          for (int pr = 0; pr < 6; ++pr)
#pragma unroll
            for (int kb = 0; kb < 4; ++kb) {
              umma_ts(tmem_wg + hn * 64, tmem_wg + 128 + pa[pr] * 32 + kb * 8,
                      b_desc_ex(w_saddr + TC_W23_BASE + pb[pr] * TC_W23_SPLIT + kb * 4096 + hn * 1024, 2048, 128), accum);
              accum = 1;
            }
          umma_commit(hn == 0 ? &S.mma_bar[wg_u] : &S.mma2_bar[wg_u]);
        }
      }
      __syncwarp();
    }
    // mean aggregation of msg at the destination nodes (:280-283): 4 threads per channel, each a run of nodes
    auto aggregate = [&](bool deg10) {
      const int c = q & 63, part = q >> 6;
      const float* col = W.stage + c;
      if (deg10) {  // same sums, no row_ptr lookups
        int nd = (nn * part) >> 2, nd1 = (nn * (part + 1)) >> 2;
        if (nn * 3 <= 64) {   // threads 192..255 hold the coordinate update: the other three quarters share the nodes
          nd = (nn * part) / 3;
          nd1 = part < 3 ? (nn * (part + 1)) / 3 : nd;
        }
        for (; nd < nd1; ++nd) {
          const float* cr = col + nd * 10 * TC_LD;
          float s0 = 0.f, s1 = 0.f;
#pragma unroll
          for (int j = 0; j < 10; j += 2) {
            s0 += cr[j * TC_LD];
            s1 += cr[(j + 1) * TC_LD];
          }
          aggr[(long)(n0 + nd) * 64 + c] = (s0 + s1) / 10.f;
        }
      } else {
        for (int nd = (nn * part) >> 2, nd1 = (nn * (part + 1)) >> 2; nd < nd1; ++nd) {
          const int rs = W.rp[buf][nd] - e0, re = W.rp[buf][nd + 1] - e0;
          float s0 = 0.f, s1 = 0.f;
          int rr = rs;
          for (; rr + 1 < re; rr += 2) {
            s0 += col[rr * TC_LD];
            s1 += col[(rr + 1) * TC_LD];
          }
          if (rr < re) s0 += col[rr * TC_LD];
          aggr[(long)(n0 + nd) * 64 + c] = re > rs ? (s0 + s1) / (float)(re - rs) : 0.f;
        }
      }
    };
    if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 12);
    mbar_wait(&S.mma_bar[wg], mma_phase);
    mma_phase ^= 1;
    tc_fence_after();
    if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 13);
    {
      float v[32];
      tmem_ld32f(d_col, v);                       // msg half row -> my own row of the (warp-private until now) tile
#pragma unroll
      for (int c = 0; c < 32; c += 2) {
        const float2 t = __fadd2_rn(f2(v[c], v[c + 1]), f2(cst.b2[half * 32 + c], cst.b2[half * 32 + c + 1]));
        v[c] = t.x; v[c + 1] = t.y;
      }
      float4* ms = reinterpret_cast<float4*>(&W.stage[r * TC_LD + half * 32]);
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) ms[c4] = make_float4(v[c4 * 4], v[c4 * 4 + 1], v[c4 * 4 + 2], v[c4 * 4 + 3]);
      mbar_wait(&S.mma2_bar[wg], mma2_phase);
      mma2_phase ^= 1;
      if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 14);
      tc_fence_after();
      tmem_ld32f(d_col + 64, v);                  // coordinate-MLP hidden half row
      float ph4[4] = {0.f, 0.f, 0.f, 0.f};        // 4 independent chains; the two halves are combined in fp64
      {
        float2 p01 = f2(0.f, 0.f), p23 = f2(0.f, 0.f);
        const float2 sl2 = f2(slope, slope);
        unsigned keep = 0;
        if (DROPOUT) keep = dropout_keep32(drop, dropout_key(drop), 8 * half, (unsigned)(e0 + r), drop.c2 + 1);
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          float2 x01 = __fadd2_rn(f2(v[c], v[c + 1]), f2(cst.b3[half * 32 + c], cst.b3[half * 32 + c + 1]));
          float2 x23 = __fadd2_rn(f2(v[c + 2], v[c + 3]), f2(cst.b3[half * 32 + c + 2], cst.b3[half * 32 + c + 3]));
          float2 y01 = __fmul2_rn(x01, sl2), y23 = __fmul2_rn(x23, sl2);
          float2 t01 = f2(fmaxf(x01.x, y01.x), fmaxf(x01.y, y01.y)), t23 = f2(fmaxf(x23.x, y23.x), fmaxf(x23.y, y23.y));
          if (DROPOUT) {   // site 1: lrelu(z3) before the w4 dot product
            t01 = __fmul2_rn(t01, f2(dropout_mul(keep, c + 0, drop.scale), dropout_mul(keep, c + 1, drop.scale)));
            t23 = __fmul2_rn(t23, f2(dropout_mul(keep, c + 2, drop.scale), dropout_mul(keep, c + 3, drop.scale)));
          }
          p01 = __ffma2_rn(t01, f2(cst.w4[half * 32 + c], cst.w4[half * 32 + c + 1]), p01);
          p23 = __ffma2_rn(t23, f2(cst.w4[half * 32 + c + 2], cst.w4[half * 32 + c + 3]), p23);
        }
        ph4[0] = p01.x; ph4[1] = p01.y; ph4[2] = p23.x; ph4[3] = p23.y;
      }
      W.red[r * 2 + half] = ((double)ph4[0] + (double)ph4[1]) + ((double)ph4[2] + (double)ph4[3]);
    }
    cp_async_wait<0>();  // next tile's indices have landed (issued behind GEMM1)
    tc_fence_before();
    // msg tile, phi halves, x_rel complete; next tile's indices visible.  The barrier also tells whether every node of the tile
    // has exactly 10 in-edges (the k-NN graphs of protein_utils.py:339-346): the tail then runs without row_ptr lookups.
    const bool deg10 = wg_barrier_and(wg, q >= nn || W.rp[buf][q + 1] - W.rp[buf][q] == 10);
    if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, tile, 15);
    // coordinate update :264, 274-277, 286-292 on the LAST threads of the group (warp 0 also issues the MMAs; the threads
    // 192..255 take no aggregation work below when all 3 nn outputs fit there)
    for (int o = 255 - q; o < nn * 3; o += 256) {
      int nd = o / 3, comp = o - nd * 3;
      int rs = W.rp[buf][nd] - e0, re = W.rp[buf][nd + 1] - e0;
      long gi = (long)(n0 + nd) * 3 + comp;
      const double xo_ = x_orig[gi], xi_ = x_in[gi];   // issued before the phi sums, consumed after them
      double sum = 0.0;
      if (deg10) {   // fixed in-degree: the same fused multiply-add chain, unrolled (its shared loads go out together)
#pragma unroll
        for (int j = 0; j < 10; ++j) {
          const int rr = nd * 10 + j;
          const double ph = W.red[rr * 2] + W.red[rr * 2 + 1] + (double)p.b_coor2;
          sum += W.xm[rr * 3 + comp] * ph;
        }
      } else
      for (int rr = rs; rr < re; ++rr) {
        const double ph = W.red[rr * 2] + W.red[rr * 2 + 1] + (double)p.b_coor2;
        sum += W.xm[rr * 3 + comp] * ph;  // x_rel * phi :264
      }
      int deg = re - rs;
      double upd = deg > 0 ? sum / (double)deg : 0.0;
      double eta = (double)p.x_connection_init;
      x_out[gi] = eta * xo_ + (1.0 - eta) * xi_ + upd;
    }
    aggregate(deg10);
    e0 = e0n; ne = nen; off_l = off_ln; n_l = n_ln; off_r = off_rn; buf ^= 1;
  }
  if (q == 0) TRACE_PHASE(0, blockIdx.x * 2 + wg, 0xffff, 16);
  cp_async_wait<0>();
  tc_fence_before();
  __syncthreads();
  TRACE_END(0);
  tmem_release(S.tmem_base, warp);
}

}  // namespace eqd

EQD_TRACE_SETTER(eqd_trace_set_edge)

namespace eqd {
int edge_stage_tc(const eqd_graph* g, const eqd_layer* p_l, const float* proj, const double* x_in, const double* x_orig,
                  float* aggr, double* x_out, int32_t* status, const DropoutArgs* drop, void* stream) {
  const eqd_layer_params* p = p_l ? &p_l->dev : nullptr;
  if (!g || !p || !proj || !x_in || !x_orig || !aggr || !x_out || !status) return EQD_ERR_BAD_ARG;
  if (!p->w_edge_tc) return EQD_ERR_BAD_ARG;
  if (g->max_in_degree < 1 || g->max_in_degree > EQD_TM) return EQD_ERR_UNSUPPORTED;
  if (!(p->leaky_slope >= 0.f && p->leaky_slope <= 1.f)) return EQD_ERR_UNSUPPORTED;  // lrelu() = max(v, slope*v)
  if ((reinterpret_cast<uintptr_t>(g->he_lig) | reinterpret_cast<uintptr_t>(g->he_rec) |
       reinterpret_cast<uintptr_t>(p->w_edge_tc)) & 15)
    return EQD_ERR_BAD_ARG;  // bulk copies need 16-byte aligned bases
  if (g->n_nodes <= 0) return EQD_OK;
  int tn = EQD_TM / g->max_in_degree;
  if (tn > TC_MAX_TN) tn = TC_MAX_TN;
  int ntiles = (g->n_nodes + tn - 1) / tn;
  EdgeConsts cst;
  memcpy(&cst, p_l->consts.edge, sizeof(cst));
  size_t smem = sizeof(TcSmem) + 128;
  int grid = (ntiles + 1) / 2;
  if (grid > 148) grid = 148;
  if (drop) {
    EQD_SET_SMEM((eqd::edge_stage_tc_kernel<true>), smem);
    eqd::edge_stage_tc_kernel<true><<<grid, TC_THREADS, smem, (cudaStream_t)stream>>>(*g, *p, cst, proj, x_in, x_orig, aggr,
                                                                                     x_out, status, tn, *drop);
  } else {
    EQD_SET_SMEM((eqd::edge_stage_tc_kernel<false>), smem);
    eqd::edge_stage_tc_kernel<false><<<grid, TC_THREADS, smem, (cudaStream_t)stream>>>(*g, *p, cst, proj, x_in, x_orig, aggr,
                                                                                      x_out, status, tn, DropoutArgs{});
  }
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}
}  // namespace eqd

extern "C" int eqd_edge_stage(const eqd_graph* g, const eqd_layer* p_l, const float* proj, const double* x_in,
                              const double* x_orig, float* aggr, double* x_out, int32_t* status, void* stream) {
  return eqd::edge_stage_tc(g, p_l, proj, x_in, x_orig, aggr, x_out, status, nullptr, stream);
}
