// Node MLP of a 64-wide IEGMN layer (rigid_docking_model.py:319-337) on the tensor cores (tcgen05, bf16x6):
//   h' = skip( W6 . LayerNorm(LeakyReLU(W5 . [h | aggr_msg | mu | h0] + b5)) + b6 )
// Weight-stationary (W5: 64x272, W6: 64x64 as bf16x3 UMMA panels, 126 KB in shared memory), two tile groups of
// 256 threads (2 threads per node row) running out of phase.  The 272-wide input is fed in 5 K-pieces.
#include "tc_common.cuh"
#include "dropout.cuh"

namespace eqd {

#define NM_THREADS 512
#define NM_W5_SPLIT 34816   // 64 x 272 bf16
#define NM_W6_BASE 104448
#define NM_W6_SPLIT 8192
#define NM_W_BYTES 129024

struct NmConsts { float b5[64], ln_g[64], ln_b[64], b6[64]; };

#define NM_SC_LD 36   // padded row stride (floats) of a warp's 32 x 32 transposition scratch: conflict-free both ways

struct NmSmem {
  unsigned char w[NM_W_BYTES];
  float sc[NM_THREADS / 32][32 * NM_SC_LD];   // one 32-row x 128-byte scratch per warp (its rows x its column half)
  float red[2][EQD_TM * 4];
  unsigned long long w_bar, a_bar[2][2];
  unsigned int tmem_base;
};

// DROPOUT (training, dropout.cuh): site 2 (node_mlp, c2 = drop.c2), mask x scale after the LeakyReLU of u5, before the
// LayerNorm statistics; 8 Philox calls per thread give the keep bits of its 32 columns.
template <bool DROPOUT>
__global__ void __launch_bounds__(NM_THREADS, 1)
node_mlp_tc_kernel(int n_nodes, eqd_layer_params p, const __grid_constant__ NmConsts cst, const float* __restrict__ h_in,
                   const float* __restrict__ aggr, const float* __restrict__ mu, const float* __restrict__ h0,
                   float* __restrict__ h_out, DropoutArgs drop) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  NmSmem& S = *reinterpret_cast<NmSmem*>(smem_raw);
  const int tid = threadIdx.x, wg = tid >> 8, q = tid & 255, half = q >> 7, r = q & 127, warp = tid >> 5;
  const int ntiles = (n_nodes + EQD_TM - 1) / EQD_TM;
  TRACE_START(3);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    mbar_init(&S.w_bar, 1);
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) mbar_init(&S.a_bar[a][b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(&S.w_bar, NM_W_BYTES);
    bulk_g2s(S.w, p.w_node_tc, NM_W_BYTES, &S.w_bar);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int wg_u = warp_u >> 3;
  const bool issuer_warp = (warp_u & 7) == 0;
  const unsigned tmem_wg = __shfl_sync(0xffffffffu, S.tmem_base, 0) + (unsigned)wg_u * 256;
  const unsigned tmem = tmem_wg + ((unsigned)((warp & 3) * 32) << 16);
  // columns: D 0..63, A 64..159
  const unsigned w_saddr = smem_u32(S.w);
  mbar_wait(&S.w_bar, 0);
  unsigned ph[2] = {0, 0};
  const float slope = p.leaky_slope;
  float* red = S.red[wg];

  // MMAs of K-blocks [kb0, kb0+nkb) of W5 (or all of W6) reading A buffer `ab`, then arrive on a_bar[ab]
  auto issue = [&](int ab, unsigned w_off, unsigned w_split, int nkb, unsigned accum0) {
    if (issuer_warp) {
      tc_fence_after();
      if (elect_one()) {
        issue_gemm(tmem_wg, tmem_wg + 64 + ab * 96, 32, w_saddr + w_off, w_split, nkb, accum0);
        umma_commit(&S.a_bar[wg_u][ab]);
      }
      __syncwarp();
    }
  };
  auto wait_a = [&](int ab) {
    mbar_wait(&S.a_bar[wg][ab], ph[ab]);
    ph[ab] ^= 1;
    tc_fence_after();
  };

  // Global rows travel coalesced: the warp's 32 rows x 128 bytes (its column half) are cp.async'ed into its scratch,
  // 8 lanes per row, one piece ahead of its use; each thread then picks up its own row.
  const int lane = tid & 31, wrow0 = 32 * (warp & 3);
  float* sc = S.sc[warp];
  auto fetch = [&](const float* base, int ld, int t) {
    if (t >= ntiles) return;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = i * 4 + (lane >> 3);
      const long nd = (long)t * EQD_TM + wrow0 + row;
      const bool ok = nd < n_nodes;   // src-size 0 zero-fills
      cp_async16(sc + row * NM_SC_LD + (lane & 7) * 4, base + (ok ? nd : 0) * ld + half * 32 + (lane & 7) * 4, ok);
    }
    cp_async_commit();
  };
  auto take = [&](float (&v)[32]) {
    cp_async_wait<0>();
    __syncwarp();
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
      float4 t = *reinterpret_cast<const float4*>(sc + lane * NM_SC_LD + c4 * 4);
      v[c4 * 4] = t.x; v[c4 * 4 + 1] = t.y; v[c4 * 4 + 2] = t.z; v[c4 * 4 + 3] = t.w;
    }
    __syncwarp();
  };
  fetch(h_in, EQD_HID, blockIdx.x * 2 + wg);
  for (int tile = blockIdx.x * 2 + wg; tile < ntiles; tile += gridDim.x * 2) {
    if (q == 0) TRACE_PHASE(3, blockIdx.x * 2 + wg, tile, 1);
    const int node = tile * EQD_TM + r;
    const bool valid = node < n_nodes;
    // ---- node_mlp.0 over [h | aggr | mu | h0] in 5 K-pieces ---------------------------------------------------
    // The tensor core truncates (round-toward-zero) on every add into an fp32 accumulator: a bias that grows with
    // the number of accumulation steps.  Each 64-wide piece is therefore its own accumulation (4 full-magnitude
    // steps, like the edge-stage GEMMs) and the pieces are summed in registers with round-to-nearest FADDs.
    float acc[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) acc[c] = cst.b5[half * 32 + c];
    {
      float v[32];
      take(v);
      fetch(aggr, EQD_HID, tile);
      store_half_split3(tmem + 64 + half * 16, v);         // piece 0 (h) -> A
    }
    tc_fence_before();
    wg_barrier(wg);
    issue(0, 0, NM_W5_SPLIT, 4, 0);
    {
      float v[32], d[32];
      auto drain = [&]() {                                  // D of the finished piece -> acc
        wait_a(0);
        tmem_ld32f(tmem + half * 32, d);
#pragma unroll
        for (int c = 0; c < 32; ++c) acc[c] += d[c];
      };
      take(v);
      fetch(mu, EQD_HID, tile);
      drain();
      store_half_split3(tmem + 64 + half * 16, v);         // piece 1 (aggr)
      tc_fence_before();
      wg_barrier(wg);
      issue(0, 4 * 2048, NM_W5_SPLIT, 4, 0);
      take(v);
      fetch(h0, EQD_H0_PAD, tile);
      drain();
      store_half_split3(tmem + 64 + half * 16, v);         // piece 2 (mu)
      tc_fence_before();
      wg_barrier(wg);
      issue(0, 8 * 2048, NM_W5_SPLIT, 4, 0);
      take(v);
      drain();
      store_half_split3(tmem + 64 + half * 16, v);         // piece 3 (h0[0:64])
      tc_fence_before();
      wg_barrier(wg);
      issue(0, 12 * 2048, NM_W5_SPLIT, 4, 0);
      drain();
      // piece 4: h0[64:72] + 8 zero columns (K = 16): the half-0 threads write 8 columns per split
      if (half == 0) {
        float t[16];
        const float4* sp = reinterpret_cast<const float4*>(h0 + (long)node * EQD_H0_PAD + 64);
        float4 a = valid ? sp[0] : make_float4(0.f, 0.f, 0.f, 0.f), b = valid ? sp[1] : make_float4(0.f, 0.f, 0.f, 0.f);
        t[0] = a.x; t[1] = a.y; t[2] = a.z; t[3] = a.w; t[4] = b.x; t[5] = b.y; t[6] = b.z; t[7] = b.w;
#pragma unroll
        for (int c = 8; c < 16; ++c) t[c] = 0.f;
        unsigned p0[8], p1[8], p2[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) split3_pair(t[2 * c], t[2 * c + 1], p0[c], p1[c], p2[c]);
        tmem_st8(tmem + 64, p0);
        tmem_st8(tmem + 64 + 32, p1);
        tmem_st8(tmem + 64 + 64, p2);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      }
      tc_fence_before();
      wg_barrier(wg);
      issue(0, 16 * 2048, NM_W5_SPLIT, 1, 0);
      drain();
    }
    // ---- + bias, LeakyReLU, LayerNorm -> bf16x3 -> A1 ; node_mlp.4 ---------------------------------------------
    {
      float v[32];
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
      unsigned keep = 0;
      if (DROPOUT) keep = dropout_keep32(drop, dropout_key(drop), 8 * half, (unsigned)node, drop.c2);
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        v[c] = lrelu(acc[c], slope);
        if (DROPOUT) v[c] *= dropout_mul(keep, c, drop.scale);
        s4[c & 3] += v[c];
      }
      const float mh = ((s4[0] + s4[1]) + (s4[2] + s4[3])) * (1.f / 32.f);
      float q4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        float d = v[c] - mh;
        q4[c & 3] = fmaf(d, d, q4[c & 3]);
      }
      red[(r * 2 + half) * 2 + 0] = mh;
      red[(r * 2 + half) * 2 + 1] = (q4[0] + q4[1]) + (q4[2] + q4[3]);
      tc_fence_before();
      wg_barrier(wg);
      const float m0 = red[r * 4 + 0], m1 = red[r * 4 + 2];
      const float mean = 0.5f * (m0 + m1);
      const float dm = m0 - m1;
      const float var = (red[r * 4 + 1] + red[r * 4 + 3] + dm * dm * 16.f) * (1.f / 64.f);  // Chan et al. combination
      const float rstd = 1.f / sqrtf(var + 1e-5f);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = (v[c] - mean) * rstd * cst.ln_g[half * 32 + c] + cst.ln_b[half * 32 + c];
      store_half_split3(tmem + 64 + half * 16, v);
    }
    tc_fence_before();
    wg_barrier(wg);
    issue(0, NM_W6_BASE, NM_W6_SPLIT, 4, 0);
    fetch(h_in, EQD_HID, tile);   // the skip operand again (an L2 hit) rather than 32 registers held across the tile
    wait_a(0);
    {
      float v[32], hskip[32];
      take(hskip);
      tmem_ld32f(tmem + half * 32, v);
      const float sk = p.skip_weight_h, sk1 = 1.f - p.skip_weight_h;
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = sk * (v[c] + cst.b6[half * 32 + c]) + sk1 * hskip[c];  // :332-334
      // transposed through the scratch: 8 lanes write one contiguous 128-byte half row
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4)
        *reinterpret_cast<float4*>(sc + lane * NM_SC_LD + c4 * 4) = make_float4(v[c4 * 4], v[c4 * 4 + 1], v[c4 * 4 + 2], v[c4 * 4 + 3]);
      __syncwarp();
      float* o = h_out + ((long)tile * EQD_TM + wrow0) * EQD_HID + half * 32 + (lane & 7) * 4;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int row = i * 4 + (lane >> 3);
        float4 t = *reinterpret_cast<const float4*>(sc + row * NM_SC_LD + (lane & 7) * 4);
        if ((long)tile * EQD_TM + wrow0 + row < n_nodes) *reinterpret_cast<float4*>(o + (long)row * EQD_HID) = t;
      }
      __syncwarp();
    }
    fetch(h_in, EQD_HID, tile + gridDim.x * 2);   // next tile's h rows, behind the end-of-tile barrier
    tc_fence_before();
    wg_barrier(wg);  // D and both A buffers are free for the next tile
  }
  tc_fence_before();
  __syncthreads();
  TRACE_END(3);
  tmem_release(S.tmem_base, warp);
}


// ---- the 69-wide layer 0 ------------------------------------------------------------------------------------------------
// h = h0 here, so the h and h0 blocks of node_mlp.0 fold into one: hidden = W5' [h0 (69 -> 80) | aggr (64) | mu (69 -> 80)]
// with N = 69 -> 80 outputs; LayerNorm over the 69 real channels; node_mlp.4 as [64][80]; no skip (widths differ, :332).
// Column ownership of the 80-wide rows: half 0 = [0,32) and the extra [64,80), half 1 = [32,64).
#define NM0_W5_SPLIT 35840    // 80 x 224 bf16
#define NM0_W6_BASE 107520
#define NM0_W6_SPLIT 10240    // 64 x 80 bf16
#define NM0_W_BYTES 138240

struct Nm0Consts { float b5[80], ln_g[80], ln_b[80], b6[64]; };

struct Nm0Smem {
  unsigned char w[NM0_W_BYTES];
  float sc[NM_THREADS / 32][32 * NM_SC_LD];
  float red[2][EQD_TM * 4];
  unsigned long long w_bar, a_bar[2];
  unsigned int tmem_base;
};

// DROPOUT: site 2 as above, on the 69 real channels (half 0 also masks the extra columns 64..68).
template <bool DROPOUT>
__global__ void __launch_bounds__(NM_THREADS, 1)
node_mlp0_tc_kernel(int n_nodes, eqd_layer_params p, const __grid_constant__ Nm0Consts cst, const float* __restrict__ h0,
                    const float* __restrict__ aggr, const float* __restrict__ mu /*[n][72]*/, float* __restrict__ h_out,
                    DropoutArgs drop) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Nm0Smem& S = *reinterpret_cast<Nm0Smem*>(smem_raw);
  const int tid = threadIdx.x, wg = tid >> 8, q = tid & 255, half = q >> 7, r = q & 127, warp = tid >> 5;
  const int ntiles = (n_nodes + EQD_TM - 1) / EQD_TM;
  TRACE_START(3);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    mbar_init(&S.w_bar, 1);
    mbar_init(&S.a_bar[0], 1);
    mbar_init(&S.a_bar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(&S.w_bar, NM0_W_BYTES);
    bulk_g2s(S.w, p.w_node_tc, NM0_W_BYTES, &S.w_bar);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int wg_u = warp_u >> 3;
  const bool issuer_warp = (warp_u & 7) == 0;
  const unsigned tmem_wg = __shfl_sync(0xffffffffu, S.tmem_base, 0) + (unsigned)wg_u * 256;
  const unsigned tmem = tmem_wg + ((unsigned)((warp & 3) * 32) << 16);
  // columns: D 0..79, A 80..199 (3 splits x 40: 32 main + 8 extra)
  const unsigned a_col = tmem + 80;
  const unsigned w_saddr = smem_u32(S.w);
  mbar_wait(&S.w_bar, 0);
  unsigned ph = 0;
  const float slope = p.leaky_slope;
  float* red = S.red[wg];

  auto issue_w5 = [&](int kb0, int nkb) {   // k-blocks [kb0, kb0 + nkb) of W5' against the A operand, fresh accumulator
    if (issuer_warp) {
      tc_fence_after();
      if (elect_one()) {
        issue_gemm_n<80>(tmem_wg, tmem_wg + 80, 40, w_saddr + kb0 * (80 * 32), NM0_W5_SPLIT, nkb);
        umma_commit(&S.a_bar[wg_u]);
      }
      __syncwarp();
    }
  };
  auto wait_a = [&]() {
    mbar_wait(&S.a_bar[wg], ph);
    ph ^= 1;
    tc_fence_after();
  };
  const int lane = tid & 31, wrow0 = 32 * (warp & 3);
  float* sc = S.sc[warp];
  auto fetch = [&](const float* base, int ld, int t) {
    if (t >= ntiles) return;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = i * 4 + (lane >> 3);
      const long nd = (long)t * EQD_TM + wrow0 + row;
      const bool ok = nd < n_nodes;   // src-size 0 zero-fills
      cp_async16(sc + row * NM_SC_LD + (lane & 7) * 4, base + (ok ? nd : 0) * ld + half * 32 + (lane & 7) * 4, ok);
    }
    cp_async_commit();
  };
  auto take = [&](float (&v)[32]) {
    cp_async_wait<0>();
    __syncwarp();
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
      float4 t = *reinterpret_cast<const float4*>(sc + lane * NM_SC_LD + c4 * 4);
      v[c4 * 4] = t.x; v[c4 * 4 + 1] = t.y; v[c4 * 4 + 2] = t.z; v[c4 * 4 + 3] = t.w;
    }
    __syncwarp();
  };
  fetch(h0, EQD_H0_PAD, blockIdx.x * 2 + wg);
  for (int tile = blockIdx.x * 2 + wg; tile < ntiles; tile += gridDim.x * 2) {
    if (q == 0) TRACE_PHASE(3, blockIdx.x * 2 + wg, tile, 1);
    const int node = tile * EQD_TM + r;
    const bool valid = node < n_nodes;
    // channels [64, 72) of an 72-strided row (zero beyond 69) as the piece's fifth k-block; half-0 threads only
    auto extra8 = [&](const float* base) {
      if (half == 0) {
        const float4* ep = reinterpret_cast<const float4*>(base + (long)node * EQD_H0_PAD + 64);
        float4 a = valid ? ep[0] : make_float4(0.f, 0.f, 0.f, 0.f), b = valid ? ep[1] : make_float4(0.f, 0.f, 0.f, 0.f);
        float t[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        store_extra8_split3(a_col + 32, t, 40);
      }
    };
    float acc[32], accx[16];   // accx: columns 64..79 (half 0)
#pragma unroll
    for (int c = 0; c < 32; ++c) acc[c] = cst.b5[half * 32 + c];
#pragma unroll
    for (int c = 0; c < 16; ++c) accx[c] = cst.b5[64 + c];
    auto drain = [&]() {   // each piece is its own accumulation (<= 5 full-magnitude steps), summed here with RN adds
      wait_a();
      float d[32];
      tmem_ld32f(tmem + half * 32, d);
#pragma unroll
      for (int c = 0; c < 32; ++c) acc[c] += d[c];
      if (half == 0) {
        float e[16];
        tmem_ld16f(tmem + 64, e);
#pragma unroll
        for (int c = 0; c < 16; ++c) accx[c] += e[c];
      }
    };
    {
      float v[32];
      take(v);
      fetch(aggr, EQD_HID, tile);
      store_half_split3(a_col + half * 16, v, 40);      // piece 0: h0 (80)
      extra8(h0);
      tc_fence_before();
      wg_barrier(wg);
      issue_w5(0, 5);
      take(v);
      fetch(mu, EQD_H0_PAD, tile);
      drain();
      store_half_split3(a_col + half * 16, v, 40);      // piece 1: aggr (64)
      tc_fence_before();
      wg_barrier(wg);
      issue_w5(5, 4);
      take(v);
      drain();
      store_half_split3(a_col + half * 16, v, 40);      // piece 2: mu (80)
      extra8(mu);
      tc_fence_before();
      wg_barrier(wg);
      issue_w5(9, 5);
      drain();
    }
    // ---- LeakyReLU, LayerNorm over the 69 real channels -> bf16x3 -> A ; node_mlp.4 ---------------------------------
    {
      const int nh = half == 0 ? 37 : 32;
      float sum = 0.f;
      unsigned keep = 0, keepx = 0;
      if (DROPOUT) {
        const unsigned long long key = dropout_key(drop);
        keep = dropout_keep32(drop, key, 8 * half, (unsigned)node, drop.c2);
        if (half == 0) keepx = dropout_keep4(drop, key, 16, (unsigned)node, drop.c2) | (dropout_keep4(drop, key, 17, (unsigned)node, drop.c2) << 4);
      }
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        acc[c] = lrelu(acc[c], slope);
        if (DROPOUT) acc[c] *= dropout_mul(keep, c, drop.scale);
        sum += acc[c];
      }
      if (half == 0) {
#pragma unroll
        for (int c = 0; c < 5; ++c) {
          accx[c] = lrelu(accx[c], slope);
          if (DROPOUT) accx[c] *= dropout_mul(keepx, c, drop.scale);
          sum += accx[c];
        }
      }
      const float mh = sum / (float)nh;
      float m2 = 0.f;
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        float d = acc[c] - mh;
        m2 = fmaf(d, d, m2);
      }
      if (half == 0) {
#pragma unroll
        for (int c = 0; c < 5; ++c) {
          float d = accx[c] - mh;
          m2 = fmaf(d, d, m2);
        }
      }
      red[(r * 2 + half) * 2 + 0] = mh;
      red[(r * 2 + half) * 2 + 1] = m2;
      tc_fence_before();
      wg_barrier(wg);
      const float m0 = red[r * 4 + 0], m1 = red[r * 4 + 2];
      const float mean = (37.f * m0 + 32.f * m1) * (1.f / 69.f);
      const float dm = m0 - m1;
      const float var = (red[r * 4 + 1] + red[r * 4 + 3] + dm * dm * (37.f * 32.f / 69.f)) * (1.f / 69.f);  // Chan et al.
      const float rstd = 1.f / sqrtf(var + 1e-5f);
#pragma unroll
      for (int c = 0; c < 32; ++c) acc[c] = (acc[c] - mean) * rstd * cst.ln_g[half * 32 + c] + cst.ln_b[half * 32 + c];
      store_half_split3(a_col + half * 16, acc, 40);
      if (half == 0) {
        float t[8];
#pragma unroll
        for (int c = 0; c < 5; ++c) t[c] = (accx[c] - mean) * rstd * cst.ln_g[64 + c] + cst.ln_b[64 + c];
        t[5] = t[6] = t[7] = 0.f;
        store_extra8_split3(a_col + 32, t, 40);
      }
    }
    tc_fence_before();
    wg_barrier(wg);
    if (issuer_warp) {
      tc_fence_after();
      if (elect_one()) {
        issue_gemm_n<64>(tmem_wg, tmem_wg + 80, 40, w_saddr + NM0_W6_BASE, NM0_W6_SPLIT, 5);
        umma_commit(&S.a_bar[wg_u]);
      }
      __syncwarp();
    }
    wait_a();
    {
      float v[32];
      tmem_ld32f(tmem + half * 32, v);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] += cst.b6[half * 32 + c];
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4)
        *reinterpret_cast<float4*>(sc + lane * NM_SC_LD + c4 * 4) = make_float4(v[c4 * 4], v[c4 * 4 + 1], v[c4 * 4 + 2], v[c4 * 4 + 3]);
      __syncwarp();
      float* o = h_out + ((long)tile * EQD_TM + wrow0) * EQD_HID + half * 32 + (lane & 7) * 4;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int row = i * 4 + (lane >> 3);
        float4 t = *reinterpret_cast<const float4*>(sc + row * NM_SC_LD + (lane & 7) * 4);
        if ((long)tile * EQD_TM + wrow0 + row < n_nodes) *reinterpret_cast<float4*>(o + (long)row * EQD_HID) = t;
      }
      __syncwarp();
    }
    fetch(h0, EQD_H0_PAD, tile + gridDim.x * 2);
    tc_fence_before();
    wg_barrier(wg);
  }
  tc_fence_before();
  __syncthreads();
  TRACE_END(3);
  tmem_release(S.tmem_base, warp);
}

}  // namespace eqd

EQD_TRACE_SETTER(eqd_trace_set_mlp)

namespace eqd {
int node_mlp_tc(const eqd_graph* g, const eqd_layer* p_l, const float* h_in, const float* aggr, const float* mu,
                const float* h0, float* h_out, const DropoutArgs* drop, void* stream) {
  const eqd_layer_params* p = p_l ? &p_l->dev : nullptr;
  if (!g || !p || !h_in || !aggr || !mu || !h0 || !h_out) return EQD_ERR_BAD_ARG;
  if (p->dh != 64 || p->dhp != 64) return EQD_ERR_UNSUPPORTED;
  if (!(p->leaky_slope >= 0.f && p->leaky_slope <= 1.f)) return EQD_ERR_UNSUPPORTED;  // lrelu() = max(v, slope*v)
  if (!p->w_node_tc || (reinterpret_cast<uintptr_t>(p->w_node_tc) & 15)) return EQD_ERR_BAD_ARG;
  if (g->n_nodes <= 0) return EQD_OK;
  NmConsts cst;
  memcpy(&cst, p_l->consts.node, sizeof(cst));
  int ntiles = (g->n_nodes + EQD_TM - 1) / EQD_TM;
  size_t smem = sizeof(NmSmem) + 128;
  int grid = (ntiles + 1) / 2;
  if (grid > 148) grid = 148;
  if (drop) {
    EQD_SET_SMEM((node_mlp_tc_kernel<true>), smem);
    node_mlp_tc_kernel<true><<<grid, NM_THREADS, smem, (cudaStream_t)stream>>>(g->n_nodes, *p, cst, h_in, aggr, mu, h0, h_out,
                                                                              *drop);
  } else {
    EQD_SET_SMEM((node_mlp_tc_kernel<false>), smem);
    node_mlp_tc_kernel<false><<<grid, NM_THREADS, smem, (cudaStream_t)stream>>>(g->n_nodes, *p, cst, h_in, aggr, mu, h0, h_out,
                                                                               DropoutArgs{});
  }
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}

int node_mlp_tc0(const eqd_graph* g, const eqd_layer* p_l, const float* h0, const float* aggr, const float* mu,
                 float* h_out, const DropoutArgs* drop, void* stream) {
  const eqd_layer_params* p = p_l ? &p_l->dev : nullptr;
  if (!g || !p || !h0 || !aggr || !mu || !h_out) return EQD_ERR_BAD_ARG;
  if (p->dh != 69 || p->dhp != 72) return EQD_ERR_UNSUPPORTED;
  if (!(p->leaky_slope >= 0.f && p->leaky_slope <= 1.f)) return EQD_ERR_UNSUPPORTED;  // lrelu() = max(v, slope*v)
  if (!p->w_node_tc || (reinterpret_cast<uintptr_t>(p->w_node_tc) & 15)) return EQD_ERR_BAD_ARG;
  if (g->n_nodes <= 0) return EQD_OK;
  Nm0Consts cst;
  memcpy(&cst, p_l->consts.node, sizeof(cst));
  int ntiles = (g->n_nodes + EQD_TM - 1) / EQD_TM;
  size_t smem = sizeof(Nm0Smem) + 128;
  int grid = (ntiles + 1) / 2;
  if (grid > 148) grid = 148;
  if (drop) {
    EQD_SET_SMEM((node_mlp0_tc_kernel<true>), smem);
    node_mlp0_tc_kernel<true><<<grid, NM_THREADS, smem, (cudaStream_t)stream>>>(g->n_nodes, *p, cst, h0, aggr, mu, h_out, *drop);
  } else {
    EQD_SET_SMEM((node_mlp0_tc_kernel<false>), smem);
    node_mlp0_tc_kernel<false><<<grid, NM_THREADS, smem, (cudaStream_t)stream>>>(g->n_nodes, *p, cst, h0, aggr, mu, h_out,
                                                                                DropoutArgs{});
  }
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}
}  // namespace eqd

extern "C" int eqd_node_mlp_tc(const eqd_graph* g, const eqd_layer* p_l, const float* h_in, const float* aggr,
                               const float* mu, const float* h0, float* h_out, void* stream) {
  return eqd::node_mlp_tc(g, p_l, h_in, aggr, mu, h0, h_out, nullptr, stream);
}

extern "C" int eqd_node_mlp_tc0(const eqd_graph* g, const eqd_layer* p_l, const float* h0, const float* aggr,
                                const float* mu, float* h_out, void* stream) {
  return eqd::node_mlp_tc0(g, p_l, h0, aggr, mu, h_out, nullptr, stream);
}

extern "C" int eqd_attention_tc0(const eqd_graph*, const float*, const void*, const float*, float*, void*);

// Layer 0 (dh == 69): attention (64 tensor-core channels + 5 fp32 ones), node MLP, next layer's projections.
namespace eqd {
int node_stage_tc0(const eqd_graph* g, const eqd_layer* p_l, const eqd_layer* p_next_l, const float* h0, const float* proj,
                   const float* aggr, void* kv, const float* x5, float* mu, float* h_out, float* proj_next,
                   const DropoutArgs* drop, void* stream) {
  const eqd_layer_params* p = p_l ? &p_l->dev : nullptr;
  const eqd_layer_params* p_next = p_next_l ? &p_next_l->dev : nullptr;
  if (!g || !p || !kv || !mu || !x5) return EQD_ERR_BAD_ARG;
  if (p_next && !proj_next) return EQD_ERR_BAD_ARG;
  int rc = eqd_attention_tc0(g, proj, kv, x5, mu, stream);
  if (rc) return rc;
  rc = node_mlp_tc0(g, p_l, h0, aggr, mu, h_out, drop, stream);
  if (rc) return rc;
  if (p_next) rc = eqd_project_tc(g, p_next_l, h_out, proj_next, kv, stream);
  return rc;
}
}  // namespace eqd

extern "C" int eqd_node_stage_tc0(const eqd_graph* g, const eqd_layer* p_l, const eqd_layer* p_next_l,
                                  const float* h0, const float* proj, const float* aggr, void* kv, const float* x5,
                                  float* mu, float* h_out, float* proj_next, void* stream) {
  return eqd::node_stage_tc0(g, p_l, p_next_l, h0, proj, aggr, kv, x5, mu, h_out, proj_next, nullptr, stream);
}

extern "C" int eqd_project_tc(const eqd_graph*, const eqd_layer*, const float*, float*, void*, void*);
extern "C" int eqd_attention_tc(const eqd_graph*, const float*, const void*, float*, void*);

namespace eqd {
int node_stage_tc(const eqd_graph* g, const eqd_layer* p_l, const eqd_layer* p_next_l, const float* h_in, const float* h0,
                  const float* proj, const float* aggr, void* kv, float* mu, float* h_out, float* proj_next,
                  const DropoutArgs* drop, void* stream) {
  const eqd_layer_params* p = p_l ? &p_l->dev : nullptr;
  const eqd_layer_params* p_next = p_next_l ? &p_next_l->dev : nullptr;
  if (!g || !p || !kv || !mu) return EQD_ERR_BAD_ARG;
  if (p_next && !proj_next) return EQD_ERR_BAD_ARG;
  int rc = eqd_attention_tc(g, proj, kv, mu, stream);
  if (rc) return rc;
  rc = node_mlp_tc(g, p_l, h_in, aggr, mu, h0, h_out, drop, stream);
  if (rc) return rc;
  if (p_next) rc = eqd_project_tc(g, p_next_l, h_out, proj_next, kv, stream);
  return rc;
}
}  // namespace eqd

extern "C" int eqd_node_stage_tc(const eqd_graph* g, const eqd_layer* p_l, const eqd_layer* p_next_l,
                                 const float* h_in, const float* h0, const float* proj, const float* aggr, void* kv,
                                 float* mu, float* h_out, float* proj_next, void* stream) {
  return eqd::node_stage_tc(g, p_l, p_next_l, h_in, h0, proj, aggr, kv, mu, h_out, proj_next, nullptr, stream);
}
