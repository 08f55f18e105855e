// Backward of the node update of IEGMN_Layer.forward (rigid_docking_model.py:319-337):
//   h' = skip( W6 . LN(LeakyReLU(W5 . [h | aggr | mu | h0] + b5)) + b6 )
// One CTA per tile of 128 nodes: recompute u5, LeakyReLU, LayerNorm statistics from the stashed inputs; then
//   do  = skH * dh'          (skip :332-334; layer 0 has none)
//   dn  = do . W6            -> LayerNorm backward -> du = da * lrelu'(u5)
//   d[h | aggr | mu | h0] = du . W5
// Outputs: dh (N x dhp, = (1-skH) dh' + h-block), daggr (N x 64), dmu (N x dhp), dh0 += h0-block (N x 72), and the
// operands of the weight-gradient reductions (n5 = LN output, du) plus per-CTA partials of dgamma / dbeta.
// Restated in oracle/backward_manual.py::node_mlp_bwd.
#include "bwd_common.cuh"
#include "dropout.cuh"

namespace eqd {

template <bool EXTRA>
struct NodeBwdCfg {
  static constexpr int DHP = EXTRA ? 72 : 64;
  static constexpr int LD = DHP + 4;
  static constexpr int BUF = EQD_TM * LD;
  static constexpr int WB = 2 * EQD_WCHUNK * EQD_WLD;
  static constexpr size_t SMEM = (size_t)(3 * BUF + WB + 16 * 64 + EQD_TM) * sizeof(float);
};

// DROPOUT: the forward's site-2 mask (c2 = drop.c2) regenerated per (node, column group): a5 = m s lrelu(u5),
// du = m s lrelu'(u5) da.
template <bool EXTRA, bool DROPOUT>
__global__ void __launch_bounds__(EQD_THREADS)
bwd_node_mlp_kernel(int n_nodes, eqd_layer_params p, const float* __restrict__ w_node1_lin /*[dhp][2dhp+136]*/,
                    const float* __restrict__ w_node2_lin /*[64][dhp]*/, const float* __restrict__ h_in, int ldh,
                    const float* __restrict__ aggr, const float* __restrict__ mu, int ldmu,
                    const float* __restrict__ h0, const float* __restrict__ dh_out, float* __restrict__ dh_in,
                    float* __restrict__ daggr, float* __restrict__ dmu, float* __restrict__ dh0_acc,
                    float* __restrict__ n5_out, float* __restrict__ du_out, float* __restrict__ vec_partial,
                    DropoutArgs drop) {
  using C = NodeBwdCfg<EXTRA>;
  constexpr int DHP = C::DHP, LD = C::LD;
  extern __shared__ __align__(16) float smem[];
  float* bufA = smem;                 // staging of the input blocks / A operand
  float* bufB = smem + C::BUF;        // second staging buffer
  float* bufH = smem + 2 * C::BUF;    // n-hat (LayerNorm normalised activations)
  float* wbuf = smem + 3 * C::BUF;
  float* scratch = wbuf + C::WB;      // 16 x 64
  float* rstd_s = scratch + 16 * 64;  // [128]
  const int tid = threadIdx.x, ty = tid >> 3, tx = tid & 7;
  const int win = 2 * DHP + 64 + EQD_H0_PAD;       // padded input width of W5 (row blocks h | aggr | mu | h0)
  const float slope = p.leaky_slope;
  const bool skip = (p.dh == EQD_HID);
  const float sk = skip ? p.skip_weight_h : 1.f;
  const bool xvalid = EXTRA && (64 + tx < p.dh);
  float gsum[8], bsum[8], gsumx = 0.f, bsumx = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) gsum[j] = bsum[j] = 0.f;

  const int ntiles = (n_nodes + EQD_TM - 1) / EQD_TM;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int node0 = tile * EQD_TM;
    const int nvalid = min(EQD_TM, n_nodes - node0);
    // ---------------- recompute u5 = W5 . [h | aggr | mu | h0] + b5 ----------------
    const float* w5 = p.w_node1;
    float acc[8][8], accx[8];
    acc_set_bias(acc, p.b_node1, tx);
#pragma unroll
    for (int i = 0; i < 8; ++i) accx[i] = EXTRA ? p.b_node1[64 + tx] : 0.f;
    tile_load_async(bufA, LD, h_in + (long)node0 * ldh, ldh, EQD_TM, nvalid, DHP, tid);
    tile_load_async(bufB, LD, mu + (long)node0 * ldmu, ldmu, EQD_TM, nvalid, DHP, tid);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    gemm_nn_stream<EXTRA>(acc, accx, bufA + ty * 8 * LD, LD, DHP, w5, DHP, DHP, wbuf, tid);
    gemm_nn_stream<EXTRA>(acc, accx, bufB + ty * 8 * LD, LD, DHP, w5 + (long)(DHP + 64) * DHP, DHP, DHP, wbuf, tid);
    tile_load_async(bufA, LD, aggr + (long)node0 * 64, 64, EQD_TM, nvalid, 64, tid);
    constexpr int H0C = EXTRA ? EQD_H0_PAD : 64;   // a 64-wide layer's tiles (LD 68) take h0 as 64 + 8 columns
    tile_load_async(bufB, LD, h0 + (long)node0 * EQD_H0_PAD, EQD_H0_PAD, EQD_TM, nvalid, H0C, tid);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    gemm_nn_stream<EXTRA>(acc, accx, bufA + ty * 8 * LD, LD, 64, w5 + (long)DHP * DHP, DHP, DHP, wbuf, tid);
    gemm_nn_stream<EXTRA>(acc, accx, bufB + ty * 8 * LD, LD, H0C, w5 + (long)(2 * DHP + 64) * DHP, DHP, DHP, wbuf, tid);
    if (!EXTRA) {
      tile_load_async(bufA, LD, h0 + (long)node0 * EQD_H0_PAD + 64, EQD_H0_PAD, EQD_TM, nvalid, 8, tid);
      cp_async_commit();
      cp_async_wait<0>();
      __syncthreads();
      gemm_nn_stream<EXTRA>(acc, accx, bufA + ty * 8 * LD, LD, 8, w5 + (long)(2 * DHP + 128) * DHP, DHP, DHP, wbuf, tid);
    }
    // ---------------- LeakyReLU + LayerNorm statistics; keep n-hat (smem), sign bits (registers) ----------------
    unsigned pos_lo = 0, pos_hi = 0, pos_x = 0;
    unsigned keep_lo = 0, keep_hi = 0, keep_x = 0;   // site-2 mask bits, same layout as pos
    const float inv_n = 1.f / (float)p.dh;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float s = 0.f;
      if (DROPOUT) {   // columns col_nn(tx, 0..7) = 4 tx + 0..3, 32 + 4 tx + 0..3; extra column 64 + tx
        const unsigned long long key = dropout_key(drop);
        const unsigned row = (unsigned)(node0 + ty * 8 + i);
        const unsigned k = dropout_keep4(drop, key, tx, row, drop.c2) | (dropout_keep4(drop, key, 8 + tx, row, drop.c2) << 4);
        if (i < 4) keep_lo |= k << (i * 8); else keep_hi |= k << ((i - 4) * 8);
        if (EXTRA) keep_x |= ((dropout_keep4(drop, key, 16 + (tx >> 2), row, drop.c2) >> (tx & 3)) & 1u) << i;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float a = lrelu(acc[i][j], slope);
        if (a > 0.f) { if (i < 4) pos_lo |= 1u << (i * 8 + j); else pos_hi |= 1u << ((i - 4) * 8 + j); }
        if (DROPOUT) a *= dropout_mul(i < 4 ? keep_lo : keep_hi, (i & 3) * 8 + j, drop.scale);
        acc[i][j] = a;
        s += a;
      }
      if (EXTRA) {
        float a = xvalid ? lrelu(accx[i], slope) : 0.f;
        if (a > 0.f) pos_x |= 1u << i;
        if (DROPOUT) a *= dropout_mul(keep_x, i, drop.scale);
        accx[i] = a;
        s += a;
      }
      float mean = row_sum8(s) * inv_n;
      float q = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float d = acc[i][j] - mean;
        q = fmaf(d, d, q);
      }
      if (EXTRA && xvalid) {
        float d = accx[i] - mean;
        q = fmaf(d, d, q);
      }
      float rstd = 1.f / sqrtf(row_sum8(q) * inv_n + 1e-5f);
      if (tx == 0) rstd_s[ty * 8 + i] = rstd;
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = (acc[i][j] - mean) * rstd;      // n-hat
      if (EXTRA) accx[i] = xvalid ? (accx[i] - mean) * rstd : 0.f;
    }
    store_tile_smem<EXTRA>(bufH, LD, acc, accx, ty, tx);
    // n5 = nhat * gamma + beta -> global (X operand of dW6 = n5^T . do)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int r = ty * 8 + i;
      if (r < nvalid) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          int c = col_nn(tx, j);
          v[j] = acc[i][j] * p.node_ln_g[c] + p.node_ln_b[c];
        }
        float* o = n5_out + (long)(node0 + r) * DHP + tx * 4;
        *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(o + 32) = make_float4(v[4], v[5], v[6], v[7]);
        if (EXTRA) n5_out[(long)(node0 + r) * DHP + 64 + tx] = xvalid ? accx[i] * p.node_ln_g[64 + tx] + p.node_ln_b[64 + tx] : 0.f;
      }
    }
    // ---------------- dn = (skH dh') . W6 ----------------
    tile_load_async(bufA, LD, dh_out + (long)node0 * 64, 64, EQD_TM, nvalid, 64, tid);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      accx[i] = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    }
    gemm_nn_stream<EXTRA>(acc, accx, bufA + ty * 8 * LD, LD, 64, w_node2_lin, DHP, DHP, wbuf, tid);
    // ---------------- LayerNorm backward, LeakyReLU backward -> du ----------------
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = ty * 8 + i;
      const float* nh = bufH + r * LD;
      float nhat[8], nhx = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        int c = col_nn(tx, j);
        nhat[j] = nh[c];
        float dn = acc[i][j] * sk;
        gsum[j] = fmaf(dn, nhat[j], gsum[j]);
        bsum[j] += dn;
        float dnh = dn * p.node_ln_g[c];
        acc[i][j] = dnh;
        s1 += dnh;
        s2 = fmaf(dnh, nhat[j], s2);
      }
      if (EXTRA) {
        nhx = nh[64 + tx];
        float dn = xvalid ? accx[i] * sk : 0.f;
        gsumx = fmaf(dn, nhx, gsumx);
        bsumx += dn;
        float dnh = xvalid ? dn * p.node_ln_g[64 + tx] : 0.f;
        accx[i] = dnh;
        s1 += dnh;
        s2 = fmaf(dnh, nhx, s2);
      }
      const float m1 = row_sum8(s1) * inv_n, m2 = row_sum8(s2) * inv_n, rstd = rstd_s[r];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        bool pos = i < 4 ? (pos_lo >> (i * 8 + j)) & 1u : (pos_hi >> ((i - 4) * 8 + j)) & 1u;
        acc[i][j] = rstd * (acc[i][j] - m1 - nhat[j] * m2) * (pos ? 1.f : slope);
        if (DROPOUT) acc[i][j] *= dropout_mul(i < 4 ? keep_lo : keep_hi, (i & 3) * 8 + j, drop.scale);
      }
      if (EXTRA) accx[i] = xvalid ? rstd * (accx[i] - m1 - nhx * m2) * (((pos_x >> i) & 1u) ? 1.f : slope) : 0.f;
      if (EXTRA && DROPOUT) accx[i] *= dropout_mul(keep_x, i, drop.scale);
    }
    __syncthreads();   // everyone is done with bufA (A operand of the W6 product)
    store_tile_smem<EXTRA>(bufA, LD, acc, accx, ty, tx);     // du: A operand of the four input-gradient products
    // du -> global (D operand of dW5 = inp^T . du, and of db5)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int r = ty * 8 + i;
      if (r < nvalid) {
        float* o = du_out + (long)(node0 + r) * DHP + tx * 4;
        *reinterpret_cast<float4*>(o) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        *reinterpret_cast<float4*>(o + 32) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
        if (EXTRA) du_out[(long)(node0 + r) * DHP + 64 + tx] = accx[i];
      }
    }
    __syncthreads();
    // ---------------- d[h | aggr | mu | h0] = du . W5 (nn.Linear layout: reduction over the hidden index) ----------------
#pragma unroll 1
    for (int blk = 0; blk < 4; ++blk) {
      const int coff = blk == 0 ? 0 : (blk == 1 ? DHP : (blk == 2 ? DHP + 64 : 2 * DHP + 64));
      const bool wide = EXTRA && blk != 1;          // 72-wide blocks: h, mu (layer 0) and h0; aggr is 64 wide
      const bool wide_h0 = !EXTRA && blk == 3;      // h0 block of a 64-wide layer: 64 + 8 columns
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        accx[i] = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
      }
      float acc2[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc2[i] = 0.f;
      if (EXTRA) {
        if (wide) gemm_nn_stream<true>(acc, accx, bufA + ty * 8 * LD, LD, DHP, w_node1_lin + coff, win, 72, wbuf, tid);
        else gemm_nn_stream<false>(acc, accx, bufA + ty * 8 * LD, LD, DHP, w_node1_lin + coff, win, 64, wbuf, tid);
      } else {
        if (wide_h0) gemm_nn_stream<true>(acc, acc2, bufA + ty * 8 * LD, LD, DHP, w_node1_lin + coff, win, 72, wbuf, tid);
        else gemm_nn_stream<false>(acc, accx, bufA + ty * 8 * LD, LD, DHP, w_node1_lin + coff, win, 64, wbuf, tid);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = ty * 8 + i;
        if (r >= nvalid) continue;
        const long n = node0 + r;
        if (blk == 0) {          // dh = (1 - skH) dh' + h block
          float add[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
          if (skip) {
            const float* d = dh_out + n * 64 + tx * 4;
            float4 a = *reinterpret_cast<const float4*>(d), b = *reinterpret_cast<const float4*>(d + 32);
            const float s1 = 1.f - p.skip_weight_h;
            add[0] = s1 * a.x; add[1] = s1 * a.y; add[2] = s1 * a.z; add[3] = s1 * a.w;
            add[4] = s1 * b.x; add[5] = s1 * b.y; add[6] = s1 * b.z; add[7] = s1 * b.w;
          }
          float* o = dh_in + n * DHP + tx * 4;
          *reinterpret_cast<float4*>(o) = make_float4(acc[i][0] + add[0], acc[i][1] + add[1], acc[i][2] + add[2], acc[i][3] + add[3]);
          *reinterpret_cast<float4*>(o + 32) = make_float4(acc[i][4] + add[4], acc[i][5] + add[5], acc[i][6] + add[6], acc[i][7] + add[7]);
          if (EXTRA) dh_in[n * DHP + 64 + tx] = accx[i];
        } else if (blk == 1) {
          float* o = daggr + n * 64 + tx * 4;
          *reinterpret_cast<float4*>(o) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
          *reinterpret_cast<float4*>(o + 32) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
        } else if (blk == 2) {
          float* o = dmu + n * DHP + tx * 4;
          *reinterpret_cast<float4*>(o) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
          *reinterpret_cast<float4*>(o + 32) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
          if (EXTRA) dmu[n * DHP + 64 + tx] = accx[i];
        } else {                 // dh0 accumulates over the layers (every node is owned by exactly one thread group)
          float* o = dh0_acc + n * EQD_H0_PAD + tx * 4;
          float4 a = *reinterpret_cast<float4*>(o), b = *reinterpret_cast<float4*>(o + 32);
          *reinterpret_cast<float4*>(o) = make_float4(a.x + acc[i][0], a.y + acc[i][1], a.z + acc[i][2], a.w + acc[i][3]);
          *reinterpret_cast<float4*>(o + 32) = make_float4(b.x + acc[i][4], b.y + acc[i][5], b.z + acc[i][6], b.w + acc[i][7]);
          dh0_acc[n * EQD_H0_PAD + 64 + tx] += EXTRA ? accx[i] : acc2[i];
        }
      }
    }
    __syncthreads();
  }
  // per-CTA partials of the LayerNorm affine gradients: vec_partial[cta][0:72] = dgamma, [72:144] = dbeta
  float* vp = vec_partial + (long)blockIdx.x * 144;
  colacc8_flush(gsum, scratch, vp, tid);
  colacc8_flush(bsum, scratch, vp + 72, tid);
  {   // channels 64..71 (layer 0 only): reduce over the 16 row groups in fixed order
    __syncthreads();
    scratch[ty * 8 + tx] = gsumx;
    scratch[128 + ty * 8 + tx] = bsumx;
    __syncthreads();
    if (tid < 8) {
      float a = 0.f, b = 0.f;
      for (int q = 0; q < 16; ++q) { a += scratch[q * 8 + tid]; b += scratch[128 + q * 8 + tid]; }
      vp[64 + tid] = a;
      vp[72 + 64 + tid] = b;
    }
  }
}

}  // namespace eqd

namespace {
template <bool EXTRA, bool DROPOUT>
int launch_bwd_node_mlp(int grid, cudaStream_t st, int n_nodes, const eqd_layer_params& p, const float* w_node1_lin,
                        const float* w_node2_lin, const float* h_in, int ldh, const float* aggr, const float* mu, int ldmu,
                        const float* h0, const float* dh_out, float* dh_in, float* daggr, float* dmu, float* dh0_acc,
                        float* n5_out, float* du_out, float* vec_partial, const eqd::DropoutArgs& d) {
  size_t smem = eqd::NodeBwdCfg<EXTRA>::SMEM;
  EQD_SET_SMEM((eqd::bwd_node_mlp_kernel<EXTRA, DROPOUT>), smem);
  eqd::bwd_node_mlp_kernel<EXTRA, DROPOUT><<<grid, EQD_THREADS, smem, st>>>(n_nodes, p, w_node1_lin, w_node2_lin, h_in, ldh,
                                                                           aggr, mu, ldmu, h0, dh_out, dh_in, daggr, dmu,
                                                                           dh0_acc, n5_out, du_out, vec_partial, d);
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}
}  // namespace

extern "C" int eqd_bwd_node_mlp(const eqd_graph* g, const eqd_layer* p_l, const float* w_node1_lin,
                                const float* w_node2_lin, const float* h_in, int32_t ldh, const float* aggr,
                                const float* mu, int32_t ldmu, const float* h0, const float* dh_out, float* dh_in,
                                float* daggr, float* dmu, float* dh0_acc, float* n5_out, float* du_out,
                                float* vec_partial, int32_t* n_partials_out, void* stream) {
  return eqd_bwd_node_mlp_dropout(g, p_l, w_node1_lin, w_node2_lin, h_in, ldh, aggr, mu, ldmu, h0, dh_out, dh_in, daggr, dmu,
                                  dh0_acc, n5_out, du_out, vec_partial, n_partials_out, nullptr, 0, stream);
}

extern "C" int eqd_bwd_node_mlp_dropout(const eqd_graph* g, const eqd_layer* p_l, const float* w_node1_lin,
                                        const float* w_node2_lin, const float* h_in, int32_t ldh, const float* aggr,
                                        const float* mu, int32_t ldmu, const float* h0, const float* dh_out, float* dh_in,
                                        float* daggr, float* dmu, float* dh0_acc, float* n5_out, float* du_out,
                                        float* vec_partial, int32_t* n_partials_out, const eqd_dropout* dropout,
                                        int32_t layer, void* stream) {
  eqd::DropoutArgs d{};
  if (const int rc = eqd::dropout_args(dropout, layer, 2, &d)) return rc;
  const eqd_layer_params* p = p_l ? &p_l->dev : nullptr;
  if (!g || !p || !w_node1_lin || !w_node2_lin || !h_in || !aggr || !mu || !h0 || !dh_out || !dh_in || !daggr || !dmu ||
      !dh0_acc || !n5_out || !du_out || !vec_partial)
    return EQD_ERR_BAD_ARG;
  const bool extra = (p->dh == 69 && p->dhp == 72);
  if (!extra && !(p->dh == 64 && p->dhp == 64)) return EQD_ERR_UNSUPPORTED;
  if (!(p->leaky_slope >= 0.f && p->leaky_slope <= 1.f)) return EQD_ERR_UNSUPPORTED;
  if ((ldh & 3) || (ldmu & 3) || ldh < p->dhp || ldmu < p->dhp) return EQD_ERR_BAD_ARG;
  const int ntiles = (g->n_nodes + EQD_TM - 1) / EQD_TM;
  int grid = ntiles < 148 ? ntiles : 148;
  if (n_partials_out) *n_partials_out = grid > 0 ? grid : 0;
  if (g->n_nodes <= 0) return EQD_OK;
  cudaStream_t st = (cudaStream_t)stream;
  auto launch = extra ? (dropout ? launch_bwd_node_mlp<true, true> : launch_bwd_node_mlp<true, false>)
                      : (dropout ? launch_bwd_node_mlp<false, true> : launch_bwd_node_mlp<false, false>);
  return launch(grid, st, g->n_nodes, *p, w_node1_lin, w_node2_lin, h_in, ldh, aggr, mu, ldmu, h0, dh_out, dh_in, daggr, dmu,
                dh0_acc, n5_out, du_out, vec_partial, d);
}
