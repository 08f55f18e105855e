// Backward of the edge stage of IEGMN_Layer.forward (rigid_docking_model.py:204-237, 263-292).
//
// bwd_edge_kernel: one CTA per tile of 128 consecutive edges.  Recomputes x_rel, the 15 RBFs, z1 = Psrc[src] + Pdst[dst]
// + W1e [he | rbf], LeakyReLU, LayerNorm, msg = W2 n + b2, z3 = W3 msg + b3, phi = w4 . lrelu(z3) + b4 from the stashed
// layer inputs, then runs the chain rule
//   dmsg_e = daggr[dst] / deg            (mean aggregation :280-283)
//   dxm_e  = dx'[dst] / deg              (mean of x_rel * phi :264, 274-277);  dphi = x_rel . dxm
//   dz3 = dphi w4 * lrelu'(z3);  dmsg += dz3 . W3;  dn = dmsg . W2;  LayerNorm backward;  dz1 = da * lrelu'(z1)
//   drbf = dz1 . W1e[:, 27:42];  d(d^2) = sum_s drbf_s rbf_s (-1/sigma_s);  dx_rel = phi dxm + 2 x_rel d(d^2)
// and leaves per-edge dz1 (E x 64), dx_rel (E x 3, fp64) and the operands of the weight-gradient reductions
// (ein = [he | rbf], n1, msg, dz3, dmsg) in HBM, plus per-CTA partials of dgamma, dbeta, dw4, db4.
// bwd_edge_gather_kernel: per node, dPsrc = sum over OUT-edges of dz1 (through the by-source permutation), dPdst = sum
// over IN-edges, dx = (1 - eta) dx' + sum_out dx_rel - sum_in dx_rel: fixed summation order, no atomics.
// Restated in oracle/backward_manual.py::edge_bwd / edge_gather.
#include "bwd_common.cuh"
#include "dropout.cuh"

namespace eqd {

#define BE_K1 44
#define BE_LD1 48
#define BE_LD 68

struct EdgeBwdSmem {
  float w1[BE_K1 * 64];        // k-major [he|rbf feature][out]
  float w2[64 * 64];           // k-major edge_mlp.4
  float w3[64 * 64];           // k-major coors_mlp.0
  float w2lin[64 * 64];        // edge_mlp.4.weight [out][in]   (k-major for dn = dmsg . W2)
  float w3lin[64 * 64];        // coors_mlp.0.weight [out][in]  (k-major for dmsg += dz3 . W3)
  float ln_g[64], ln_b[64], b2[64], b3[64], w4[64];
  float bufE[EQD_TM * BE_LD1];  // [he | rbf]
  float bufA[EQD_TM * BE_LD];   // current A operand
  float bufH[EQD_TM * BE_LD];   // n-hat
  float scratch[16 * 64];
  double xrel[EQD_TM * 3];
  double dxm[EQD_TM * 3];
  float phi[EQD_TM], dphi[EQD_TM], rstd[EQD_TM], invdeg[EQD_TM];
  int src[EQD_TM], dst[EQD_TM];
};

// DROPOUT: the forward's site-0 / site-1 masks (c2 = drop.c2, drop.c2 + 1) are regenerated per (row, column group):
// a1 = m s lrelu(z1), dz1 = m s lrelu'(z1) da;  c3 = m s lrelu(z3) (phi, dw4), dz3 = m s lrelu'(z3) dphi w4.
template <bool DROPOUT>
__global__ void __launch_bounds__(EQD_THREADS)
bwd_edge_kernel(eqd_graph g, eqd_layer_params p, const float* __restrict__ w2lin, const float* __restrict__ w3lin,
                const float* __restrict__ proj, const double* __restrict__ x_in, const float* __restrict__ daggr,
                const double* __restrict__ dx_out, float* __restrict__ ein_out, float* __restrict__ n1_out,
                float* __restrict__ msg_out, float* __restrict__ dz3_out, float* __restrict__ dmsg_out,
                float* __restrict__ dz1_out, double* __restrict__ dxrel_out, float* __restrict__ vec_partial,
                DropoutArgs drop) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  EdgeBwdSmem& s = *reinterpret_cast<EdgeBwdSmem*>(smem_raw);
  const int tid = threadIdx.x, ty = tid >> 3, tx = tid & 7;
  const int pw = 128 + 3 * p.dhp;
  const float slope = p.leaky_slope;
  for (int i = tid; i < BE_K1 * 64 / 4; i += EQD_THREADS)
    reinterpret_cast<float4*>(s.w1)[i] = reinterpret_cast<const float4*>(p.w_edge1)[i];
  for (int i = tid; i < 64 * 64 / 4; i += EQD_THREADS) {
    reinterpret_cast<float4*>(s.w2)[i] = reinterpret_cast<const float4*>(p.w_edge2)[i];
    reinterpret_cast<float4*>(s.w3)[i] = reinterpret_cast<const float4*>(p.w_coor1)[i];
    reinterpret_cast<float4*>(s.w2lin)[i] = reinterpret_cast<const float4*>(w2lin)[i];
    reinterpret_cast<float4*>(s.w3lin)[i] = reinterpret_cast<const float4*>(w3lin)[i];
  }
  if (tid < 64) {
    s.ln_g[tid] = p.edge_ln_g[tid];
    s.ln_b[tid] = p.edge_ln_b[tid];
    s.b2[tid] = p.b_edge2[tid];
    s.b3[tid] = p.b_coor1[tid];
    s.w4[tid] = p.w_coor2[tid];
  }
  __syncthreads();
  float gsum[8], bsum[8], w4sum[8], b4sum = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) gsum[j] = bsum[j] = w4sum[j] = 0.f;

  const int E = g.n_edges;
  const int ntiles = (E + EQD_TM - 1) / EQD_TM;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int e0 = tile * EQD_TM;
    const int ne = min(EQD_TM, E - e0);
    // ---- per-edge geometry and the gradient of the two mean aggregations: thread t <-> edge e0 + t ----
    {
      float* row = s.bufE + tid * BE_LD1;
      if (tid < ne) {
        const int e = e0 + tid;
        const int sn = g.col_src[e], dn = g.edge_dst[e];
        s.src[tid] = sn;
        s.dst[tid] = dn;
        const double rx = x_in[(long)sn * 3 + 0] - x_in[(long)dn * 3 + 0];
        const double ry = x_in[(long)sn * 3 + 1] - x_in[(long)dn * 3 + 1];
        const double rz = x_in[(long)sn * 3 + 2] - x_in[(long)dn * 3 + 2];
        s.xrel[tid * 3 + 0] = rx; s.xrel[tid * 3 + 1] = ry; s.xrel[tid * 3 + 2] = rz;
        const float d2 = (float)(rx * rx + ry * ry + rz * rz);
        float sigma = 1.f;
#pragma unroll
        for (int q = 0; q < EQD_N_RBF; ++q) {
          row[EQD_EDGE_FEATS + q] = expf(-d2 / sigma);
          sigma *= 1.5f;
        }
        const int deg = g.row_ptr[dn + 1] - g.row_ptr[dn];
        const double inv = deg > 0 ? 1.0 / (double)deg : 0.0;
        s.invdeg[tid] = (float)inv;
        const double mx = dx_out[(long)dn * 3 + 0] * inv, my = dx_out[(long)dn * 3 + 1] * inv, mz = dx_out[(long)dn * 3 + 2] * inv;
        s.dxm[tid * 3 + 0] = mx; s.dxm[tid * 3 + 1] = my; s.dxm[tid * 3 + 2] = mz;
        const float dph = (float)(rx * mx + ry * my + rz * mz);
        s.dphi[tid] = dph;
        b4sum += dph;
      } else {
        s.src[tid] = -1;
        s.dst[tid] = -1;
        s.invdeg[tid] = 0.f;
        s.dphi[tid] = 0.f;
#pragma unroll
        for (int q = 0; q < EQD_N_RBF; ++q) row[EQD_EDGE_FEATS + q] = 0.f;
      }
      row[42] = 0.f;
      row[43] = 0.f;
    }
    for (int idx = tid; idx < EQD_TM * EQD_EDGE_FEATS; idx += EQD_THREADS) {
      int r = idx / EQD_EDGE_FEATS, k = idx - r * EQD_EDGE_FEATS;
      float v = 0.f;
      if (r < ne) {
        int e = e0 + r;
        v = e < g.n_lig_edges ? g.he_lig[(long)e * EQD_EDGE_FEATS + k]
                              : g.he_rec[(long)(e - g.n_lig_edges) * EQD_EDGE_FEATS + k];
      }
      s.bufE[r * BE_LD1 + k] = v;
    }
    __syncthreads();
    // ein = [he | rbf | 0 0] -> global (X operand of dW1e)
    for (int idx = tid; idx < ne * (BE_K1 / 4); idx += EQD_THREADS) {
      int r = idx / (BE_K1 / 4), c4 = idx - r * (BE_K1 / 4);
      *reinterpret_cast<float4*>(ein_out + (long)(e0 + r) * BE_K1 + c4 * 4) =
          *reinterpret_cast<const float4*>(s.bufE + r * BE_LD1 + c4 * 4);
    }
    // ---- z1, LeakyReLU, LayerNorm: keep n-hat (smem), rstd (smem), sign(z1) (registers) ----
    float acc[8][8], accx[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int r = ty * 8 + i;
      int sn = s.src[r], dn = s.dst[r];
      if (sn >= 0) {
        const float* ps = proj + (long)sn * pw + tx * 4;
        const float* pd = proj + (long)dn * pw + 64 + tx * 4;
        float4 a0 = *reinterpret_cast<const float4*>(ps), a1 = *reinterpret_cast<const float4*>(ps + 32);
        float4 b0 = *reinterpret_cast<const float4*>(pd), b1 = *reinterpret_cast<const float4*>(pd + 32);
        acc[i][0] = a0.x + b0.x; acc[i][1] = a0.y + b0.y; acc[i][2] = a0.z + b0.z; acc[i][3] = a0.w + b0.w;
        acc[i][4] = a1.x + b1.x; acc[i][5] = a1.y + b1.y; acc[i][6] = a1.z + b1.z; acc[i][7] = a1.w + b1.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
      }
    }
    gemm_nn<false>(acc, accx, s.bufE + ty * 8 * BE_LD1, BE_LD1, s.w1, 64, BE_K1, tx);
    unsigned pos_lo = 0, pos_hi = 0, keep_lo = 0, keep_hi = 0;   // keep: site-0 mask bits, same layout as pos
    float nrm[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float sum = 0.f;
      if (DROPOUT) {   // columns col_nn(tx, 0..7) = 4 tx + 0..3, 32 + 4 tx + 0..3
        const unsigned long long key = dropout_key(drop);
        const unsigned row = (unsigned)(e0 + ty * 8 + i);
        const unsigned k = dropout_keep4(drop, key, tx, row, drop.c2) | (dropout_keep4(drop, key, 8 + tx, row, drop.c2) << 4);
        if (i < 4) keep_lo |= k << (i * 8); else keep_hi |= k << ((i - 4) * 8);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float a = lrelu(acc[i][j], slope);
        if (a > 0.f) { if (i < 4) pos_lo |= 1u << (i * 8 + j); else pos_hi |= 1u << ((i - 4) * 8 + j); }
        if (DROPOUT) a *= dropout_mul(i < 4 ? keep_lo : keep_hi, (i & 3) * 8 + j, drop.scale);
        acc[i][j] = a;
        sum += a;
      }
      const float mean = row_sum8(sum) * (1.f / 64.f);
      float q = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float d = acc[i][j] - mean;
        q = fmaf(d, d, q);
      }
      const float rstd = 1.f / sqrtf(row_sum8(q) * (1.f / 64.f) + 1e-5f);
      if (tx == 0) s.rstd[ty * 8 + i] = rstd;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = col_nn(tx, j);
        acc[i][j] = (acc[i][j] - mean) * rstd;                 // n-hat
        nrm[i][j] = acc[i][j] * s.ln_g[c] + s.ln_b[c];          // n1
      }
    }
    store_tile_smem<false>(s.bufH, BE_LD, acc, accx, ty, tx);
    store_tile_smem<false>(s.bufA, BE_LD, nrm, accx, ty, tx);
    store_tile_global(n1_out, e0, 64, ne, nrm, ty, tx);
    __syncthreads();
    // ---- msg = W2 n1 + b2 ----
    acc_set_bias(acc, s.b2, tx);
    gemm_nn<false>(acc, accx, s.bufA + ty * 8 * BE_LD, BE_LD, s.w2, 64, 64, tx);
    __syncthreads();
    store_tile_smem<false>(s.bufA, BE_LD, acc, accx, ty, tx);
    store_tile_global(msg_out, e0, 64, ne, acc, ty, tx);
    __syncthreads();
    // ---- z3 = W3 msg + b3, c3 = lrelu(z3), phi; dz3 = dphi w4 lrelu'(z3); dw4 += c3 dphi ----
    acc_set_bias(acc, s.b3, tx);
    gemm_nn<false>(acc, accx, s.bufA + ty * 8 * BE_LD, BE_LD, s.w3, 64, 64, tx);
    {
      float w4r[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) w4r[j] = s.w4[col_nn(tx, j)];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = ty * 8 + i;
        const float dph = s.dphi[r];
        float v = 0.f;
        unsigned keep = 0;
        if (DROPOUT) {
          const unsigned long long key = dropout_key(drop);
          const unsigned row = (unsigned)(e0 + r);
          keep = dropout_keep4(drop, key, tx, row, drop.c2 + 1) | (dropout_keep4(drop, key, 8 + tx, row, drop.c2 + 1) << 4);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float c3 = lrelu(acc[i][j], slope);
          if (DROPOUT) {
            const float m = dropout_mul(keep, j, drop.scale);
            const float c3m = c3 * m;
            v = fmaf(c3m, w4r[j], v);
            w4sum[j] = fmaf(c3m, dph, w4sum[j]);
            acc[i][j] = dph * w4r[j] * lrelu_grad_from_post(c3, slope) * m;   // dz3
          } else {
            v = fmaf(c3, w4r[j], v);
            w4sum[j] = fmaf(c3, dph, w4sum[j]);
            acc[i][j] = dph * w4r[j] * lrelu_grad_from_post(c3, slope);     // dz3
          }
        }
        v = row_sum8(v);
        if (tx == 0) s.phi[r] = v + p.b_coor2;
      }
    }
    __syncthreads();   // bufA (msg) no longer read
    store_tile_smem<false>(s.bufA, BE_LD, acc, accx, ty, tx);
    store_tile_global(dz3_out, e0, 64, ne, acc, ty, tx);
    __syncthreads();
    // ---- dmsg = daggr[dst] / deg + dz3 . W3 ----
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = ty * 8 + i;
      const int dn = s.dst[r];
      if (dn >= 0) {
        const float inv = s.invdeg[r];
        const float* d = daggr + (long)dn * 64 + tx * 4;
        float4 a = *reinterpret_cast<const float4*>(d), b = *reinterpret_cast<const float4*>(d + 32);
        acc[i][0] = a.x * inv; acc[i][1] = a.y * inv; acc[i][2] = a.z * inv; acc[i][3] = a.w * inv;
        acc[i][4] = b.x * inv; acc[i][5] = b.y * inv; acc[i][6] = b.z * inv; acc[i][7] = b.w * inv;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
      }
    }
    gemm_nn<false>(acc, accx, s.bufA + ty * 8 * BE_LD, BE_LD, s.w3lin, 64, 64, tx);
    __syncthreads();
    store_tile_smem<false>(s.bufA, BE_LD, acc, accx, ty, tx);
    store_tile_global(dmsg_out, e0, 64, ne, acc, ty, tx);
    __syncthreads();
    // ---- dn = dmsg . W2; LayerNorm backward; dz1 = da lrelu'(z1) ----
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    gemm_nn<false>(acc, accx, s.bufA + ty * 8 * BE_LD, BE_LD, s.w2lin, 64, 64, tx);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = ty * 8 + i;
      const float* nh = s.bufH + r * BE_LD;
      float nhat[8], s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = col_nn(tx, j);
        nhat[j] = nh[c];
        const float dn = acc[i][j];
        gsum[j] = fmaf(dn, nhat[j], gsum[j]);
        bsum[j] += dn;
        const float dnh = dn * s.ln_g[c];
        acc[i][j] = dnh;
        s1 += dnh;
        s2 = fmaf(dnh, nhat[j], s2);
      }
      const float m1 = row_sum8(s1) * (1.f / 64.f), m2 = row_sum8(s2) * (1.f / 64.f), rstd = s.rstd[r];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const bool pos = i < 4 ? (pos_lo >> (i * 8 + j)) & 1u : (pos_hi >> ((i - 4) * 8 + j)) & 1u;
        acc[i][j] = rstd * (acc[i][j] - m1 - nhat[j] * m2) * (pos ? 1.f : slope);
        if (DROPOUT) acc[i][j] *= dropout_mul(i < 4 ? keep_lo : keep_hi, (i & 3) * 8 + j, drop.scale);
      }
    }
    __syncthreads();   // bufA (dmsg) no longer read
    store_tile_smem<false>(s.bufA, BE_LD, acc, accx, ty, tx);
    store_tile_global(dz1_out, e0, 64, ne, acc, ty, tx);
    __syncthreads();
    // ---- coordinates: thread t <-> edge.  drbf = dz1 . W1e[rbf rows]; d(d^2); dx_rel ----
    if (tid < ne) {
      const float* dz = s.bufA + tid * BE_LD;
      float drbf[EQD_N_RBF];
#pragma unroll
      for (int q = 0; q < EQD_N_RBF; ++q) drbf[q] = 0.f;
#pragma unroll 4
      for (int n4 = 0; n4 < 16; ++n4) {
        const float4 d = *reinterpret_cast<const float4*>(dz + n4 * 4);
#pragma unroll
        for (int q = 0; q < EQD_N_RBF; ++q) {
          const float4 w = *reinterpret_cast<const float4*>(s.w1 + (EQD_EDGE_FEATS + q) * 64 + n4 * 4);
          drbf[q] = fmaf(d.x, w.x, fmaf(d.y, w.y, fmaf(d.z, w.z, fmaf(d.w, w.w, drbf[q]))));
        }
      }
      double dd2 = 0.0, sigma = 1.0;
#pragma unroll
      for (int q = 0; q < EQD_N_RBF; ++q) {
        dd2 -= (double)drbf[q] * (double)s.bufE[tid * BE_LD1 + EQD_EDGE_FEATS + q] / sigma;
        sigma *= 1.5;
      }
      const double ph = (double)s.phi[tid];
#pragma unroll
      for (int c = 0; c < 3; ++c)
        dxrel_out[(long)(e0 + tid) * 3 + c] = ph * s.dxm[tid * 3 + c] + 2.0 * s.xrel[tid * 3 + c] * dd2;
    }
    __syncthreads();
  }
  // per-CTA partials: [0:64) dgamma, [64:128) dbeta, [128:192) dw4, [192] db4
  float* vp = vec_partial + (long)blockIdx.x * 256;
  colacc8_flush(gsum, s.scratch, vp, tid);
  colacc8_flush(bsum, s.scratch, vp + 64, tid);
  colacc8_flush(w4sum, s.scratch, vp + 128, tid);
  s.scratch[tid] = b4sum;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
    for (int q = 0; q < EQD_THREADS; ++q) t += s.scratch[q];
    vp[192] = t;
  }
}

// One warp per node; lane l owns channels 2l, 2l+1 of dPsrc / dPdst and (lanes 0..2) one coordinate.
__global__ void bwd_edge_gather_kernel(eqd_graph g, const int* __restrict__ out_ptr, const int* __restrict__ out_edge,
                                       const float* __restrict__ dz1, const double* __restrict__ dxrel,
                                       const double* __restrict__ dx_out, float eta, float* __restrict__ dP, int ldp,
                                       double* __restrict__ dx_in) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= g.n_nodes) return;
  const int n = warp;
  float2 ssum = make_float2(0.f, 0.f), dsum = make_float2(0.f, 0.f);
  double cx = 0.0;
  const int i0 = g.row_ptr[n], i1 = g.row_ptr[n + 1];
  for (int e = i0; e < i1; ++e) {                 // in-edges: contiguous
    const float2 v = *reinterpret_cast<const float2*>(dz1 + (long)e * 64 + lane * 2);
    dsum.x += v.x; dsum.y += v.y;
    if (lane < 3) cx -= dxrel[(long)e * 3 + lane];
  }
  const int o0 = out_ptr[n], o1 = out_ptr[n + 1];
  for (int q = o0; q < o1; ++q) {                 // out-edges: through the by-source permutation (ascending edge id)
    const int e = out_edge[q];
    const float2 v = *reinterpret_cast<const float2*>(dz1 + (long)e * 64 + lane * 2);
    ssum.x += v.x; ssum.y += v.y;
    if (lane < 3) cx += dxrel[(long)e * 3 + lane];
  }
  *reinterpret_cast<float2*>(dP + (long)n * ldp + lane * 2) = ssum;
  *reinterpret_cast<float2*>(dP + (long)n * ldp + 64 + lane * 2) = dsum;
  if (lane < 3) dx_in[(long)n * 3 + lane] = (1.0 - (double)eta) * dx_out[(long)n * 3 + lane] + cx;
}

}  // namespace eqd

extern "C" int eqd_bwd_edge(const eqd_graph* g, const eqd_layer* p_l, const float* w2lin, const float* w3lin,
                            const float* proj, const double* x_in, const float* daggr, const double* dx_out,
                            float* ein_out, float* n1_out, float* msg_out, float* dz3_out, float* dmsg_out, float* dz1_out,
                            double* dxrel_out, float* vec_partial, int32_t* n_partials_out, void* stream) {
  return eqd_bwd_edge_dropout(g, p_l, w2lin, w3lin, proj, x_in, daggr, dx_out, ein_out, n1_out, msg_out, dz3_out, dmsg_out,
                              dz1_out, dxrel_out, vec_partial, n_partials_out, nullptr, 0, stream);
}

extern "C" int eqd_bwd_edge_dropout(const eqd_graph* g, const eqd_layer* p_l, const float* w2lin, const float* w3lin,
                                    const float* proj, const double* x_in, const float* daggr, const double* dx_out,
                                    float* ein_out, float* n1_out, float* msg_out, float* dz3_out, float* dmsg_out,
                                    float* dz1_out, double* dxrel_out, float* vec_partial, int32_t* n_partials_out,
                                    const eqd_dropout* dropout, int32_t layer, void* stream) {
  eqd::DropoutArgs d{};
  if (const int rc = eqd::dropout_args(dropout, layer, 0, &d)) return rc;
  const eqd_layer_params* p = p_l ? &p_l->dev : nullptr;
  if (!g || !p || !w2lin || !w3lin || !proj || !x_in || !daggr || !dx_out || !ein_out || !n1_out || !msg_out || !dz3_out ||
      !dmsg_out || !dz1_out || !dxrel_out || !vec_partial)
    return EQD_ERR_BAD_ARG;
  if (!(p->leaky_slope >= 0.f && p->leaky_slope <= 1.f)) return EQD_ERR_UNSUPPORTED;
  const int ntiles = (g->n_edges + EQD_TM - 1) / EQD_TM;
  int grid = ntiles < 148 ? ntiles : 148;
  if (n_partials_out) *n_partials_out = grid > 0 ? grid : 0;
  if (g->n_edges <= 0) return EQD_OK;
  size_t smem = sizeof(eqd::EdgeBwdSmem);
  if (dropout) {
    EQD_SET_SMEM((eqd::bwd_edge_kernel<true>), smem);
    eqd::bwd_edge_kernel<true><<<grid, EQD_THREADS, smem, (cudaStream_t)stream>>>(
        *g, *p, w2lin, w3lin, proj, x_in, daggr, dx_out, ein_out, n1_out, msg_out, dz3_out, dmsg_out, dz1_out, dxrel_out,
        vec_partial, d);
  } else {
    EQD_SET_SMEM((eqd::bwd_edge_kernel<false>), smem);
    eqd::bwd_edge_kernel<false><<<grid, EQD_THREADS, smem, (cudaStream_t)stream>>>(
        *g, *p, w2lin, w3lin, proj, x_in, daggr, dx_out, ein_out, n1_out, msg_out, dz3_out, dmsg_out, dz1_out, dxrel_out,
        vec_partial, d);
  }
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}

extern "C" int eqd_bwd_edge_gather(const eqd_graph* g, const int32_t* out_ptr, const int32_t* out_edge, const float* dz1,
                                   const double* dxrel, const double* dx_out, float eta, float* dP, int32_t ldp,
                                   double* dx_in, void* stream) {
  if (!g || !out_ptr || !out_edge || !dz1 || !dxrel || !dx_out || !dP || !dx_in || ldp < 128 || (ldp & 1))
    return EQD_ERR_BAD_ARG;
  if (g->n_nodes <= 0) return EQD_OK;
  const long threads = (long)g->n_nodes * 32;
  eqd::bwd_edge_gather_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      *g, out_ptr, out_edge, dz1, dxrel, dx_out, eta, dP, ldp, dx_in);
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}
