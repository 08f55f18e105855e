// Keypoint read-out + Kabsch (IEGMN.forward, rigid_docking_model.py:521-600) and the final rigid
// transform of the ligand (Rigid_Body_Docking_Net.forward :657-665).  All arithmetic after the
// mean-pooling GEMM is fp64: the 50-head softmax weights multiply last-layer coordinates that
// reach O(10^3) A, so this is where fp32 rounding would cost 1e-4 A.
//
// Algebra: the reference materialises keys (n x 3200) and compares them with the 3200-d query;
//   logits[k][j] = <W_K,k h_j , W_Q,k qbar> / sqrt(64) = h_j . u_k,   u_k = (W_K,k^T W_Q,k / 8) qbar = m_qk[k]^T qbar
// so only u (50 x 64) is formed per protein, from 50 64x64 matrices folded once per model (eqd_head_fold; SURVEY 8a
// row a9) -- 40x fewer FLOPs, same value up to rounding.
#include <cstdlib>

#include "common.cuh"
#include "svd3.cuh"
#include "dropout.cuh"

namespace eqd {

#define HEAD_THREADS 256
#define HEAD_ULD 66   // padded row stride (doubles) of u[50][64]; even: rows are read as double2
#define HEAD_HLD 66   // padded row stride (doubles) of the staged h chunk
#define HEAD_JC 64    // nodes per staged chunk

// ---- partial column sums of LeakyReLU(W_m h + b_m) over each node tile (:525, :529) -------------
// DROPOUT (training, dropout.cuh): site 3 (mlp_h_mean_ROT, c2 = drop.c2), mask x scale before the column sums.
template <bool DROPOUT>
__global__ void __launch_bounds__(EQD_THREADS, 2)
head_mean_kernel(eqd_graph g, eqd_head_params hp, const float* __restrict__ h, float* __restrict__ part, DropoutArgs drop) {
  TRACE_START(5);
  extern __shared__ __align__(16) float smem[];
  constexpr int LD = 68;
  float* A = smem;                   // [128][68]
  float* wbuf = smem + EQD_TM * LD;  // weight ring; reused as the reduction scratch [16][64]
  const int tid = threadIdx.x, ty = tid >> 3, tx = tid & 7;
  for (int tile = blockIdx.x; tile < g.n_node_tiles; tile += gridDim.x) {
    const int seg = g.node_tiles[2 * tile], node0 = g.node_tiles[2 * tile + 1];
    const int nvalid = min(EQD_TM, g.seg_ptr[seg + 1] - node0);
    tile_load_async(A, LD, h + (long)node0 * EQD_HID, EQD_HID, EQD_TM, nvalid, EQD_HID, tid);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    float acc[8][8], accx[8];
    acc_set_bias(acc, hp.b_mean, tx);
    gemm_nn_stream<false>(acc, accx, A + ty * 8 * LD, LD, EQD_HID, hp.w_mean, EQD_HID, EQD_HID, wbuf, tid);
    float colsum[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) colsum[j] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (ty * 8 + i < nvalid) {
        unsigned keep = 0;
        if (DROPOUT) {   // columns 4 tx .. 4 tx + 3 and 32 + 4 tx .. 32 + 4 tx + 3 (col_nn)
          const unsigned long long key = dropout_key(drop);
          const unsigned row = (unsigned)(node0 + ty * 8 + i);
          keep = dropout_keep4(drop, key, tx, row, drop.c2) | (dropout_keep4(drop, key, 8 + tx, row, drop.c2) << 4);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float a = lrelu(acc[i][j], hp.leaky_slope);
          if (DROPOUT) a *= dropout_mul(keep, j, drop.scale);
          colsum[j] += a;
        }
      }
#pragma unroll
    for (int j = 0; j < 8; ++j) wbuf[ty * 64 + col_nn(tx, j)] = colsum[j];
    __syncthreads();
    if (tid < 64) {
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < 16; ++q) s += wbuf[q * 64 + tid];
      part[(long)tile * 64 + tid] = s;
    }
    __syncthreads();
  }
}

// ---- batched head algebra ---------------------------------------------------------------------------------------
// qbar[s][64] = mean over segment s of LeakyReLU(W_m h + b_m)   (from the per-tile partial sums)
__global__ void head_qbar_kernel(eqd_graph g, const float* __restrict__ part, const int* __restrict__ tile_ptr,
                                 double* __restrict__ qbar) {
  int s = blockIdx.x, c = threadIdx.x;  // 64 threads
  double acc = 0.0;
  for (int t = tile_ptr[s]; t < tile_ptr[s + 1]; ++t) acc += (double)part[(long)t * 64 + c];
  int n = g.seg_ptr[s + 1] - g.seg_ptr[s];
  qbar[(long)s * 64 + c] = n > 0 ? acc / (double)n : 0.0;
}

// Weights-only fold, once per model:  m_qk[k][d'][d] = sum_e W_query[k*64+e][d'] W_key[k*64+e][d] / sqrt(64)
// so that u_k = m_qk[k]^T qbar -- the 3200-d query never has to be formed per protein.  CTA = one head.
__global__ void __launch_bounds__(256) head_fold_kernel(eqd_head_params hp, double* __restrict__ m_qk) {
  __shared__ float wq[64][65], wk[64][65];
  const int k = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < 64 * 64; i += 256) {
    wq[i >> 6][i & 63] = hp.w_query[(long)k * 4096 + i];
    wk[i >> 6][i & 63] = hp.w_key[(long)k * 4096 + i];
  }
  __syncthreads();
  const int d = tid & 63;
  for (int dq = tid >> 6; dq < 64; dq += 4) {
    double a = 0.0;
    for (int e = 0; e < 64; ++e) a = fma((double)wq[e][dq], (double)wk[e][d], a);
    m_qk[((long)k * 64 + dq) * 64 + d] = a * 0.125;  // / math.sqrt(d), d = 64 (:545)
  }
}

// u[s][k][d] = sum_d' m_qk[k][d'][d] * qbar[partner(s)][d'].  CTA = one head k (its 32 KB fold in smem) x a stripe of
// segments; a thread owns channels (lane, lane + 32) of 8 segments at a time (the qbar loads are warp-uniform
// broadcasts): 4 shared + 8 global 16-byte loads feed 32 DFMAs.
__global__ void __launch_bounds__(256) head_u_kernel(int n_pairs, const double* __restrict__ m_qk,
                                                     const double* __restrict__ qbar, double* __restrict__ u) {
  __shared__ double m[64][64];
  const int k = blockIdx.x, tid = threadIdx.x, nseg = 2 * n_pairs;
  for (int i = tid; i < 64 * 64; i += 256) m[i >> 6][i & 63] = m_qk[(long)k * 4096 + i];
  __syncthreads();
  const int lane = tid & 31, warp = tid >> 5;
  for (int s0 = blockIdx.y * 64 + warp * 8; s0 < nseg; s0 += gridDim.y * 64) {
    const double* q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int s = min(s0 + j, nseg - 1);
      int ps = s < n_pairs ? s + n_pairs : s - n_pairs;   // the query comes from the partner protein (:544, :555)
      q[j] = qbar + (long)ps * 64;
    }
    double acc[8][2];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = 0.0;
#pragma unroll 2
    for (int dd = 0; dd < 64; dd += 2) {
      const double a0 = m[dd][lane], a1 = m[dd + 1][lane], b0 = m[dd][lane + 32], b1 = m[dd + 1][lane + 32];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const double2 qv = *reinterpret_cast<const double2*>(q[j] + dd);
        acc[j][0] = fma(a1, qv.y, fma(a0, qv.x, acc[j][0]));
        acc[j][1] = fma(b1, qv.y, fma(b0, qv.x, acc[j][1]));
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (s0 + j < nseg) {
        u[((long)(s0 + j) * EQD_HEADS + k) * 64 + lane] = acc[j][0];
        u[((long)(s0 + j) * EQD_HEADS + k) * 64 + lane + 32] = acc[j][1];
      }
  }
}

// ---- keypoints: grid (segment, head half); 5 warps x 5 heads per CTA ------------------------------------------------
#define KP_HEADS_PER_CTA 25
#define KP_NH 5            // heads per warp
#define KP_THREADS 160
struct KeypSmem {
  double u[KP_HEADS_PER_CTA * HEAD_ULD];
  double hc[HEAD_JC * HEAD_HLD];  // the staged h chunk, already widened to fp64
  double xc[HEAD_JC * 3];
};

// One CTA per (protein s, 25 of the 50 heads): keypoints Y_s[k][3] (:542-560).  Warp w owns heads 25 y + 5 w + j; every
// lane keeps its OWN online-softmax state (max, sum, sum p x) per head over the rows it sees (rows lane, lane + 32 of each
// 64-row chunk), so the chunk loop has no cross-lane traffic at all; the 32 partial states are merged once at the end.
__global__ void __launch_bounds__(KP_THREADS, 4)
keypoints_kernel(eqd_graph g, const float* __restrict__ h, const double* __restrict__ x,
                 const double* __restrict__ u_all /* [2B][50][64] */, double* __restrict__ keypts) {
  TRACE_START(6);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  KeypSmem& s = *reinterpret_cast<KeypSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int seg = blockIdx.x, head0 = blockIdx.y * KP_HEADS_PER_CTA;
  const int i0 = g.seg_ptr[seg], i1 = g.seg_ptr[seg + 1];

  for (int o = tid; o < KP_HEADS_PER_CTA * 64; o += KP_THREADS)
    s.u[(o >> 6) * HEAD_ULD + (o & 63)] = u_all[((long)seg * EQD_HEADS + head0) * 64 + o];

  double m[KP_NH], l[KP_NH], sx[KP_NH], sy[KP_NH], sz[KP_NH];
#pragma unroll
  for (int j = 0; j < KP_NH; ++j) {
    m[j] = -INFINITY;
    l[j] = sx[j] = sy[j] = sz[j] = 0.0;
  }
  const double* uw = s.u + (warp * KP_NH) * HEAD_ULD;
  const double* h0r = s.hc + lane * HEAD_HLD;
  const double* h1r = s.hc + (lane + 32) * HEAD_HLD;

  for (int c0 = i0; c0 < i1; c0 += HEAD_JC) {
    const int nc = min(HEAD_JC, i1 - c0);
    __syncthreads();   // the previous chunk (and, first time round, u) is no longer / now visible
    for (int idx = tid; idx < HEAD_JC * 16; idx += KP_THREADS) {
      const int r = idx >> 4, d4 = (idx & 15) * 4;
      float4 v = r < nc ? *reinterpret_cast<const float4*>(h + (long)(c0 + r) * EQD_HID + d4) : make_float4(0.f, 0.f, 0.f, 0.f);
      double* dst = s.hc + r * HEAD_HLD + d4;
      *reinterpret_cast<double2*>(dst) = make_double2((double)v.x, (double)v.y);
      *reinterpret_cast<double2*>(dst + 2) = make_double2((double)v.z, (double)v.w);
    }
    for (int idx = tid; idx < HEAD_JC * 3; idx += KP_THREADS) s.xc[idx] = idx < nc * 3 ? x[(long)c0 * 3 + idx] : 0.0;
    __syncthreads();
    // logits of this warp's 5 heads for 2 rows: 7 16-byte shared loads feed 20 DFMAs per pair of channels
    double lg[KP_NH][2];
#pragma unroll
    for (int j = 0; j < KP_NH; ++j) lg[j][0] = lg[j][1] = 0.0;
    if (nc > 32) {
#pragma unroll 4
      for (int d = 0; d < 64; d += 2) {
        const double2 a = *reinterpret_cast<const double2*>(h0r + d), b = *reinterpret_cast<const double2*>(h1r + d);
#pragma unroll
        for (int j = 0; j < KP_NH; ++j) {
          const double2 uv = *reinterpret_cast<const double2*>(uw + j * HEAD_ULD + d);
          lg[j][0] = fma(a.y, uv.y, fma(a.x, uv.x, lg[j][0]));
          lg[j][1] = fma(b.y, uv.y, fma(b.x, uv.x, lg[j][1]));
        }
      }
    } else {   // a short last chunk: only the first row of each lane exists
#pragma unroll 4
      for (int d = 0; d < 64; d += 2) {
        const double2 a = *reinterpret_cast<const double2*>(h0r + d);
#pragma unroll
        for (int j = 0; j < KP_NH; ++j) {
          const double2 uv = *reinterpret_cast<const double2*>(uw + j * HEAD_ULD + d);
          lg[j][0] = fma(a.y, uv.y, fma(a.x, uv.x, lg[j][0]));
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int r = lane + 32 * q;
      if (r < nc) {
        const double px = s.xc[r * 3 + 0], py = s.xc[r * 3 + 1], pz = s.xc[r * 3 + 2];
#pragma unroll
        for (int j = 0; j < KP_NH; ++j) {
          const double dlt = lg[j][q] - m[j];       // +inf on the lane's first row
          const double e = exp(-fabs(dlt));
          const bool up = dlt > 0.0;
          const double pj = up ? 1.0 : e, sc = up ? e : 1.0;
          m[j] = up ? lg[j][q] : m[j];
          l[j] = fma(l[j], sc, pj);
          sx[j] = fma(sx[j], sc, pj * px);
          sy[j] = fma(sy[j], sc, pj * py);
          sz[j] = fma(sz[j], sc, pj * pz);
        }
      }
    }
  }
  // merge the 32 per-lane states of each head
#pragma unroll
  for (int j = 0; j < KP_NH; ++j) {
    const double mm = warp_max_d(m[j]);
    const double sc = m[j] == -INFINITY ? 0.0 : exp(m[j] - mm);
    const double lt = warp_sum_d(l[j] * sc), ax = warp_sum_d(sx[j] * sc), ay = warp_sum_d(sy[j] * sc), az = warp_sum_d(sz[j] * sc);
    if (lane == 0) {
      const double inv = 1.0 / lt;
      double* y = keypts + ((long)seg * EQD_HEADS + head0 + warp * KP_NH + j) * 3;
      y[0] = ax * inv;
      y[1] = ay * inv;
      y[2] = az * inv;
    }
  }
}

// One warp per pair: keypoint means and A = (Y_rec - mean)^T (Y_lig - mean)  (:563-567).
__global__ void keypoint_cov_kernel(int n_pairs, const double* __restrict__ keypts, double* __restrict__ ymean,
                                    double* __restrict__ cov) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= n_pairs) return;
  const double* yl = keypts + (long)b * EQD_HEADS * 3;
  const double* yr = keypts + (long)(n_pairs + b) * EQD_HEADS * 3;
  double ml[3], mr[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    double a = 0.0, r = 0.0;
    for (int k = lane; k < EQD_HEADS; k += 32) {
      a += yl[k * 3 + c];
      r += yr[k * 3 + c];
    }
    ml[c] = warp_sum_d(a) / (double)EQD_HEADS;
    mr[c] = warp_sum_d(r) / (double)EQD_HEADS;
  }
  double A[9];
#pragma unroll
  for (int q = 0; q < 9; ++q) A[q] = 0.0;
  for (int k = lane; k < EQD_HEADS; k += 32) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) A[r * 3 + c] += (yr[k * 3 + r] - mr[r]) * (yl[k * 3 + c] - ml[c]);
  }
#pragma unroll
  for (int q = 0; q < 9; ++q) A[q] = warp_sum_d(A[q]);
  if (lane == 0) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      ymean[(long)b * 3 + c] = ml[c];
      ymean[(long)(n_pairs + b) * 3 + c] = mr[c];
    }
#pragma unroll
    for (int q = 0; q < 9; ++q) cov[(long)b * 9 + q] = A[q];
  }
}

// One CTA per pair: thread 0 solves Kabsch (:571-589), then all threads move that pair's ligand (:665).
__global__ void kabsch_apply_kernel(eqd_graph g, const double* __restrict__ cov, const double* __restrict__ ymean,
                                    const float* __restrict__ x_lig_in, const int* __restrict__ pair_mask,
                                    float* __restrict__ rot, float* __restrict__ trans, float* __restrict__ ligand_out,
                                    double* __restrict__ sing, int* __restrict__ status) {
  TRACE_START(7);
  const int b = blockIdx.x;
  if (pair_mask && pair_mask[b] == 0) return;
  __shared__ double Tb[12];
  if (threadIdx.x == 0) {
    double A[9], U[9], S[3], V[9];
    bool nan = false;
#pragma unroll
    for (int q = 0; q < 9; ++q) {
      A[q] = cov[(long)b * 9 + q];
      nan |= !(A[q] == A[q]);
    }
    svd3(A, U, S, V);
    int st = 0;
    if (nan) st |= EQD_STATUS_NAN;
    // guard of :574, evaluated on the fp32-rounded singular values like the reference's fp32 S
    {
      float s0 = (float)S[0], s1 = (float)S[1], s2 = (float)S[2];
      float q0 = s0 * s0, q1 = s1 * s1, q2 = s2 * s2;
      float gap = fminf(fminf(fabsf(q0 - q1), fabsf(q0 - q2)), fabsf(q1 - q2));
      if (fminf(fminf(s0, s1), s2) < 1e-3f || gap < 1e-2f) st |= EQD_STATUS_SVD_DEGENERATE;
    }
    double det = A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) +
                 A[2] * (A[3] * A[7] - A[4] * A[6]);
    double sg = det > 0.0 ? 1.0 : (det < 0.0 ? -1.0 : 0.0);  // torch.sign(torch.det(A)) :586
    const double* ml = ymean + (long)b * 3;
    const double* mr = ymean + (long)(g.n_pairs + b) * 3;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
      for (int c = 0; c < 3; ++c)  // T = U diag(1,1,sg) V^T :587
        Tb[r * 3 + c] = U[r * 3 + 0] * V[c * 3 + 0] + U[r * 3 + 1] * V[c * 3 + 1] + sg * U[r * 3 + 2] * V[c * 3 + 2];
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)  // b = mean_rec - T mean_lig :589
      Tb[9 + r] = mr[r] - (Tb[r * 3 + 0] * ml[0] + Tb[r * 3 + 1] * ml[1] + Tb[r * 3 + 2] * ml[2]);
#pragma unroll
    for (int q = 0; q < 9; ++q) rot[(long)b * 9 + q] = (float)Tb[q];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      trans[(long)b * 3 + q] = (float)Tb[9 + q];
      sing[(long)b * 3 + q] = S[q];
    }
    status[b] = st;
  }
  __syncthreads();
  const int i0 = g.seg_ptr[b], i1 = g.seg_ptr[b + 1];
  for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
    double px = (double)x_lig_in[(long)i * 3 + 0], py = (double)x_lig_in[(long)i * 3 + 1],
           pz = (double)x_lig_in[(long)i * 3 + 2];
#pragma unroll
    for (int r = 0; r < 3; ++r)
      ligand_out[(long)i * 3 + r] = (float)(Tb[r * 3 + 0] * px + Tb[r * 3 + 1] * py + Tb[r * 3 + 2] * pz + Tb[9 + r]);
  }
}

// tile_ptr[s] = index of the first node tile of segment s (tiles are emitted segment by segment)
__global__ void tile_ptr_kernel(eqd_graph g, int* __restrict__ tile_ptr) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  int nseg = 2 * g.n_pairs;
  if (s > nseg) return;
  if (s == nseg) {
    tile_ptr[s] = g.n_node_tiles;
    return;
  }
  // binary search for the first tile whose segment >= s
  int lo = 0, hi = g.n_node_tiles;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (g.node_tiles[2 * mid] < s) lo = mid + 1; else hi = mid;
  }
  tile_ptr[s] = lo;
}

}  // namespace eqd

EQD_TRACE_SETTER(eqd_trace_set_head)

static inline size_t eqd_align256(size_t v) { return (v + 255) & ~(size_t)255; }

extern "C" int eqd_abi_version(void) { return EQD_ABI_VERSION; }

static inline size_t ws_part_bytes(int32_t n_node_tiles) { return eqd_align256((size_t)(n_node_tiles > 0 ? n_node_tiles : 1) * 64 * sizeof(float)); }
static inline size_t ws_tile_ptr_bytes(int32_t n_pairs) { return eqd_align256((size_t)(2 * (n_pairs > 0 ? n_pairs : 0) + 1) * sizeof(int)); }
static inline size_t ws_qbar_bytes(int32_t n_pairs) { return eqd_align256((size_t)2 * (n_pairs > 0 ? n_pairs : 1) * 64 * sizeof(double)); }
static inline size_t ws_u_bytes(int32_t n_pairs) { return eqd_align256((size_t)2 * (n_pairs > 0 ? n_pairs : 1) * EQD_HEADS * 64 * sizeof(double)); }

extern "C" size_t eqd_workspace_bytes(int32_t n_nodes, int32_t n_node_tiles, int32_t n_pairs) {
  (void)n_nodes;
  // per-tile partial sums | first tile of each segment | qbar[2B][64] | u[2B][50][64]   (fp64 from qbar on)
  return ws_part_bytes(n_node_tiles) + ws_tile_ptr_bytes(n_pairs) + ws_qbar_bytes(n_pairs) + ws_u_bytes(n_pairs);
}

extern "C" int eqd_head_fold(const eqd_head_params* hp, double* m_qk, void* stream) {
  if (!hp || !hp->w_key || !hp->w_query || !m_qk) return EQD_ERR_BAD_ARG;
  eqd::head_fold_kernel<<<EQD_HEADS, 256, 0, (cudaStream_t)stream>>>(*hp, m_qk);
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}

namespace eqd {
int keypoints(const eqd_graph* g, const eqd_head_params* hp, const float* h, const double* x, void* workspace,
              size_t workspace_bytes, double* keypts, double* ymean, double* cov, const DropoutArgs* drop, void* stream) {
  if (!g || !hp || !h || !x || !workspace || !keypts || !ymean || !cov) return EQD_ERR_BAD_ARG;
  if (!hp->m_qk || (reinterpret_cast<uintptr_t>(hp->m_qk) & 15)) return EQD_ERR_BAD_ARG;   // eqd_head_fold() output
  if (workspace_bytes < eqd_workspace_bytes(g->n_nodes, g->n_node_tiles, g->n_pairs)) return EQD_ERR_WORKSPACE;
  if (!(hp->leaky_slope >= 0.f && hp->leaky_slope <= 1.f)) return EQD_ERR_UNSUPPORTED;
  if (g->n_pairs <= 0) return EQD_OK;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* wsb = reinterpret_cast<unsigned char*>(workspace);
  float* part = reinterpret_cast<float*>(wsb);
  int* tile_ptr = reinterpret_cast<int*>(wsb + ws_part_bytes(g->n_node_tiles));
  double* qbar = reinterpret_cast<double*>(wsb + ws_part_bytes(g->n_node_tiles) + ws_tile_ptr_bytes(g->n_pairs));
  double* u = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(qbar) + ws_qbar_bytes(g->n_pairs));
  const int nseg = 2 * g->n_pairs;
  {
    size_t smem = (size_t)(EQD_TM * 68 + 2 * EQD_WCHUNK * EQD_WLD) * sizeof(float);
    int grid = g->n_node_tiles < 148 * 2 ? g->n_node_tiles : 148 * 2;
    if (drop) {
      EQD_SET_SMEM((eqd::head_mean_kernel<true>), smem);
      eqd::head_mean_kernel<true><<<grid, EQD_THREADS, smem, st>>>(*g, *hp, h, part, *drop);
    } else {
      EQD_SET_SMEM((eqd::head_mean_kernel<false>), smem);
      eqd::head_mean_kernel<false><<<grid, EQD_THREADS, smem, st>>>(*g, *hp, h, part, DropoutArgs{});
    }
    EQD_CUDA_LAUNCH_CHECK();
  }
  {
    eqd::tile_ptr_kernel<<<(nseg + 1 + 127) / 128, 128, 0, st>>>(*g, tile_ptr);
    EQD_CUDA_LAUNCH_CHECK();
    eqd::head_qbar_kernel<<<nseg, 64, 0, st>>>(*g, part, tile_ptr, qbar);
    EQD_CUDA_LAUNCH_CHECK();
    int gy = (nseg + 63) / 64;
    if (gy > 8) gy = 8;
    eqd::head_u_kernel<<<dim3(EQD_HEADS, gy), 256, 0, st>>>(g->n_pairs, hp->m_qk, qbar, u);
    EQD_CUDA_LAUNCH_CHECK();
  }
  {
    size_t smem = sizeof(eqd::KeypSmem);
    EQD_SET_SMEM((eqd::keypoints_kernel), smem);
    eqd::keypoints_kernel<<<dim3(2 * g->n_pairs, EQD_HEADS / KP_HEADS_PER_CTA), KP_THREADS, smem, st>>>(*g, h, x, u, keypts);
    EQD_CUDA_LAUNCH_CHECK();
  }
  {
    int warps_per_block = 4;
    int grid = (g->n_pairs + warps_per_block - 1) / warps_per_block;
    eqd::keypoint_cov_kernel<<<grid, warps_per_block * 32, 0, st>>>(g->n_pairs, keypts, ymean, cov);
    EQD_CUDA_LAUNCH_CHECK();
  }
  return EQD_OK;
}
}  // namespace eqd

extern "C" int eqd_keypoints(const eqd_graph* g, const eqd_head_params* hp, const float* h, const double* x,
                             void* workspace, size_t workspace_bytes, double* keypts, double* ymean, double* cov,
                             void* stream) {
  return eqd::keypoints(g, hp, h, x, workspace, workspace_bytes, keypts, ymean, cov, nullptr, stream);
}

extern "C" int eqd_kabsch_apply(const eqd_graph* g, const double* cov, const double* ymean, const float* x_lig_in,
                                const int32_t* pair_mask, float* rot, float* trans, float* ligand_out, double* sing,
                                int32_t* status, void* stream) {
  if (!g || !cov || !ymean || !x_lig_in || !rot || !trans || !ligand_out || !sing || !status) return EQD_ERR_BAD_ARG;
  if (g->n_pairs <= 0) return EQD_OK;
  eqd::kabsch_apply_kernel<<<g->n_pairs, 128, 0, (cudaStream_t)stream>>>(*g, cov, ymean, x_lig_in, pair_mask, rot,
                                                                        trans, ligand_out, sing, status);
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}

// =====================================================================================================================
// BACKWARD of the keypoint read-out and the Kabsch step (no code in the reference: what loss.backward(), train.py:154,
// makes of rigid_docking_model.py:521-589, 657-665).  fp64 throughout; every reduction in a fixed order.  Restated in
// oracle/backward_manual.py::kabsch_bwd / svd_rotation_backward / keypoints_bwd.
// =====================================================================================================================
namespace eqd {

// One CTA per pair.  coords = T new_x + b (:665), b = ym_r - T ym_l (:589), T = U D V^T with D = diag(1,1,sign det A) a
// constant (:586-587), A = (Y_r - ym_r)^T (Y_l - ym_l) (:567).  gA = U [ (skew(U^T gU)/E) S + S (skew(V^T gV)/E) ] V^T with
// gU = gT V D, gV = gT^T U D, E_jk = S_k^2 - S_j^2 (torch's svd_backward; |E| >= 1e-2 is what the guard :574 enforces).
__global__ void __launch_bounds__(128)
kabsch_bwd_kernel(eqd_graph g, const double* __restrict__ cov, const double* __restrict__ ymean,
                  const double* __restrict__ keypts, const float* __restrict__ x_lig_in, const float* __restrict__ dcoors,
                  const double* __restrict__ dY_direct, const float* __restrict__ drot, const float* __restrict__ dtrans,
                  double* __restrict__ dY) {
  const int b = blockIdx.x, tid = threadIdx.x, B = g.n_pairs;
  __shared__ double red[128][12];
  __shared__ double dA[9], dyml[3], dymr[3];
  const int i0 = g.seg_ptr[b], i1 = g.seg_ptr[b + 1];
  double acc[12];
#pragma unroll
  for (int q = 0; q < 12; ++q) acc[q] = 0.0;
  if (dcoors) {
    for (int i = i0 + tid; i < i1; i += 128) {
      const double gx = dcoors[(long)i * 3], gy = dcoors[(long)i * 3 + 1], gz = dcoors[(long)i * 3 + 2];
      const double px = x_lig_in[(long)i * 3], py = x_lig_in[(long)i * 3 + 1], pz = x_lig_in[(long)i * 3 + 2];
      acc[0] += gx * px; acc[1] += gx * py; acc[2] += gx * pz;
      acc[3] += gy * px; acc[4] += gy * py; acc[5] += gy * pz;
      acc[6] += gz * px; acc[7] += gz * py; acc[8] += gz * pz;
      acc[9] += gx; acc[10] += gy; acc[11] += gz;
    }
  }
#pragma unroll
  for (int q = 0; q < 12; ++q) red[tid][q] = acc[q];
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1) {
    if (tid < s)
#pragma unroll
      for (int q = 0; q < 12; ++q) red[tid][q] += red[tid + s][q];
    __syncthreads();
  }
  if (tid == 0) {
    double gT[9], gb[3], A[9], U[9], S[3], V[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) gT[q] = red[0][q] + (drot ? (double)drot[(long)b * 9 + q] : 0.0);
#pragma unroll
    for (int q = 0; q < 3; ++q) gb[q] = red[0][9 + q] + (dtrans ? (double)dtrans[(long)b * 3 + q] : 0.0);
#pragma unroll
    for (int q = 0; q < 9; ++q) A[q] = cov[(long)b * 9 + q];
    svd3(A, U, S, V);
    const double det = A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) +
                       A[2] * (A[3] * A[7] - A[4] * A[6]);
    const double sg = det > 0.0 ? 1.0 : (det < 0.0 ? -1.0 : 0.0);
    const double Dg[3] = {1.0, 1.0, sg};
    const double* ml = ymean + (long)b * 3;
    const double* mr = ymean + (long)(B + b) * 3;
    double T[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c)
        T[r * 3 + c] = U[r * 3] * V[c * 3] + U[r * 3 + 1] * V[c * 3 + 1] + sg * U[r * 3 + 2] * V[c * 3 + 2];
    // b = ym_r - T ym_l
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      dymr[r] = gb[r];
      dyml[r] = -(T[0 * 3 + r] * gb[0] + T[1 * 3 + r] * gb[1] + T[2 * 3 + r] * gb[2]);
#pragma unroll
      for (int c = 0; c < 3; ++c) gT[r * 3 + c] -= gb[r] * ml[c];
    }
    // gU = gT V D ; gV = gT^T U D
    double gU[9], gV[9], P[9], Q[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        gU[r * 3 + c] = (gT[r * 3] * V[0 * 3 + c] + gT[r * 3 + 1] * V[1 * 3 + c] + gT[r * 3 + 2] * V[2 * 3 + c]) * Dg[c];
        gV[r * 3 + c] = (gT[0 * 3 + r] * U[0 * 3 + c] + gT[1 * 3 + r] * U[1 * 3 + c] + gT[2 * 3 + r] * U[2 * 3 + c]) * Dg[c];
      }
    // P = U^T gU, Q = V^T gV
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        P[r * 3 + c] = U[0 * 3 + r] * gU[0 * 3 + c] + U[1 * 3 + r] * gU[1 * 3 + c] + U[2 * 3 + r] * gU[2 * 3 + c];
        Q[r * 3 + c] = V[0 * 3 + r] * gV[0 * 3 + c] + V[1 * 3 + r] * gV[1 * 3 + c] + V[2 * 3 + r] * gV[2 * 3 + c];
      }
    double In[9];
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        if (j == k) { In[j * 3 + k] = 0.0; continue; }
        const double E = S[k] * S[k] - S[j] * S[j];
        In[j * 3 + k] = ((P[j * 3 + k] - P[k * 3 + j]) / E) * S[k] + S[j] * ((Q[j * 3 + k] - Q[k * 3 + j]) / E);
      }
    // gA = U In V^T
    double UI[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) UI[r * 3 + c] = U[r * 3] * In[0 * 3 + c] + U[r * 3 + 1] * In[1 * 3 + c] + U[r * 3 + 2] * In[2 * 3 + c];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) dA[r * 3 + c] = UI[r * 3] * V[c * 3] + UI[r * 3 + 1] * V[c * 3 + 1] + UI[r * 3 + 2] * V[c * 3 + 2];
  }
  __syncthreads();
  // dYc_r = Yc_l dA^T, dYc_l = Yc_r dA; un-centre: dY = dYc - mean_k(dYc) + dym / K
  __shared__ double dyc[2][EQD_HEADS][3];
  const double* ml = ymean + (long)b * 3;
  const double* mr = ymean + (long)(B + b) * 3;
  const double* yl = keypts + (long)b * EQD_HEADS * 3;
  const double* yr = keypts + (long)(B + b) * EQD_HEADS * 3;
  if (tid < EQD_HEADS) {
    const int k = tid;
    const double cl[3] = {yl[k * 3] - ml[0], yl[k * 3 + 1] - ml[1], yl[k * 3 + 2] - ml[2]};
    const double cr[3] = {yr[k * 3] - mr[0], yr[k * 3 + 1] - mr[1], yr[k * 3 + 2] - mr[2]};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      dyc[1][k][c] = cl[0] * dA[c * 3 + 0] + cl[1] * dA[c * 3 + 1] + cl[2] * dA[c * 3 + 2];   // (Yc_l dA^T)[k][c]
      dyc[0][k][c] = cr[0] * dA[0 * 3 + c] + cr[1] * dA[1 * 3 + c] + cr[2] * dA[2 * 3 + c];   // (Yc_r dA)[k][c]
    }
  }
  __syncthreads();
  __shared__ double mean_d[2][3];
  if (tid < 6) {
    const int side = tid / 3, c = tid % 3;
    double t = 0.0;
    for (int k = 0; k < EQD_HEADS; ++k) t += dyc[side][k][c];
    mean_d[side][c] = t / (double)EQD_HEADS;
  }
  __syncthreads();
  for (int o = tid; o < 2 * EQD_HEADS * 3; o += 128) {
    const int side = o / (EQD_HEADS * 3), rem = o - side * EQD_HEADS * 3, k = rem / 3, c = rem - k * 3;
    const long gi = ((long)(side == 0 ? b : B + b) * EQD_HEADS + k) * 3 + c;
    double v = dyc[side][k][c] - mean_d[side][c] + (side == 0 ? dyml[c] : dymr[c]) / (double)EQD_HEADS;
    if (dY_direct) v += dY_direct[gi];
    dY[gi] = v;
  }
}

// logits[n][k] = h_n . u[seg(n)][k]   (warp per node, lanes over heads)
__global__ void kp_logits_kernel(eqd_graph g, const int* __restrict__ node_seg, const float* __restrict__ h,
                                 const double* __restrict__ u, double* __restrict__ logits) {
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (n >= g.n_nodes) return;
  const int s = node_seg[n];
  const float* hr = h + (long)n * EQD_HID;
  for (int k = lane; k < EQD_HEADS; k += 32) {
    const double* uk = u + ((long)s * EQD_HEADS + k) * 64;
    double t = 0.0;
#pragma unroll 8
    for (int d = 0; d < 64; ++d) t = fma((double)hr[d], uk[d], t);
    logits[(long)n * EQD_HEADS + k] = t;
  }
}

// per (segment, head): softmax statistics over the segment's nodes and c_k = dY_k . Y_k.  stats[s][k] = {m, 1/l, c}
__global__ void kp_stats_kernel(eqd_graph g, const double* __restrict__ logits, const double* __restrict__ keypts,
                                const double* __restrict__ dY, double* __restrict__ stats) {
  const int s = blockIdx.x, k = threadIdx.x;
  if (k >= EQD_HEADS) return;
  const int i0 = g.seg_ptr[s], i1 = g.seg_ptr[s + 1];
  double m = -INFINITY;
  for (int i = i0; i < i1; ++i) m = fmax(m, logits[(long)i * EQD_HEADS + k]);
  double l = 0.0;
  for (int i = i0; i < i1; ++i) l += exp(logits[(long)i * EQD_HEADS + k] - m);
  const double* y = keypts + ((long)s * EQD_HEADS + k) * 3;
  const double* d = dY + ((long)s * EQD_HEADS + k) * 3;
  double* o = stats + ((long)s * EQD_HEADS + k) * 3;
  o[0] = m;
  o[1] = l > 0.0 ? 1.0 / l : 0.0;
  o[2] = d[0] * y[0] + d[1] * y[1] + d[2] * y[2];
}

// warp per node n: att_k = exp(logit - m_k) / l_k; dlog_k = att_k (dY_k . z_n - c_k) (overwrites logits[n][k]);
// dz_n = sum_k att_k dY_k -> dx[n];  dh[n][d] = sum_k dlog_k u_k[d]
__global__ void kp_node_bwd_kernel(eqd_graph g, const int* __restrict__ node_seg, const double* __restrict__ x,
                                   const double* __restrict__ u, const double* __restrict__ dY,
                                   const double* __restrict__ stats, double* __restrict__ logits,
                                   double* __restrict__ dx, float* __restrict__ dh) {
  __shared__ double dl[8][EQD_HEADS + 2];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x * 8 + w;
  if (n < g.n_nodes) {
    const int s = node_seg[n];
    const double zx = x[(long)n * 3], zy = x[(long)n * 3 + 1], zz = x[(long)n * 3 + 2];
    double ax = 0.0, ay = 0.0, az = 0.0;
    for (int k = lane; k < EQD_HEADS; k += 32) {
      const double* st = stats + ((long)s * EQD_HEADS + k) * 3;
      const double* d = dY + ((long)s * EQD_HEADS + k) * 3;
      const double att = exp(logits[(long)n * EQD_HEADS + k] - st[0]) * st[1];
      const double dlog = att * (d[0] * zx + d[1] * zy + d[2] * zz - st[2]);
      logits[(long)n * EQD_HEADS + k] = dlog;
      dl[w][k] = dlog;
      ax += att * d[0]; ay += att * d[1]; az += att * d[2];
    }
    ax = warp_sum_d(ax); ay = warp_sum_d(ay); az = warp_sum_d(az);
    if (lane == 0) { dx[(long)n * 3] = ax; dx[(long)n * 3 + 1] = ay; dx[(long)n * 3 + 2] = az; }
    __syncwarp();
    double a0 = 0.0, a1 = 0.0;
    for (int k = 0; k < EQD_HEADS; ++k) {
      const double* uk = u + ((long)s * EQD_HEADS + k) * 64;
      a0 = fma(dl[w][k], uk[lane], a0);
      a1 = fma(dl[w][k], uk[lane + 32], a1);
    }
    dh[(long)n * EQD_HID + lane] = (float)a0;
    dh[(long)n * EQD_HID + lane + 32] = (float)a1;
  }
}

// du[s][k][d] = sum_{n in seg s} dlog[n][k] h[n][d]   (CTA per segment, fixed order over n)
__global__ void __launch_bounds__(256) kp_du_kernel(eqd_graph g, const double* __restrict__ dlog, const float* __restrict__ h,
                                                    double* __restrict__ du) {
  const int s = blockIdx.x, i0 = g.seg_ptr[s], i1 = g.seg_ptr[s + 1];
  for (int o = threadIdx.x; o < EQD_HEADS * 64; o += 256) {
    const int k = o >> 6, d = o & 63;
    double t = 0.0;
    for (int i = i0; i < i1; ++i) t = fma(dlog[(long)i * EQD_HEADS + k], (double)h[(long)i * EQD_HID + d], t);
    du[(long)s * EQD_HEADS * 64 + o] = t;
  }
}

// CTA per head k: over all segments s (fixed order): r = W_Q,k qbar_partner(s), a = W_K,k du_{s,k} / 8,
// dW_K,k[e][d] += r[e] du[d] / 8, dW_Q,k[e][d'] += a[e] qbar_partner[d'].  a is kept for the dqbar pass.
__global__ void __launch_bounds__(256)
head_weight_bwd_kernel(int n_pairs, eqd_head_params hp, const double* __restrict__ qbar, const double* __restrict__ du,
                       double* __restrict__ a_out /*[2B][50][64]*/, float* __restrict__ g_wkey, float* __restrict__ g_wquery) {
  __shared__ float wq[64][65], wk[64][65];
  __shared__ double r[64], a[64], qb[64], dv[64];
  const int k = blockIdx.x, tid = threadIdx.x, nseg = 2 * n_pairs;
  for (int i = tid; i < 64 * 64; i += 256) {
    wq[i >> 6][i & 63] = hp.w_query[(long)k * 4096 + i];
    wk[i >> 6][i & 63] = hp.w_key[(long)k * 4096 + i];
  }
  double gk[16], gq[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) gk[q] = gq[q] = 0.0;
  const int e0 = (tid >> 6) * 16, d = tid & 63;      // this thread owns (e0 .. e0+15, d)
  for (int s = 0; s < nseg; ++s) {
    const int ps = s < n_pairs ? s + n_pairs : s - n_pairs;
    __syncthreads();
    if (tid < 64) {
      qb[tid] = qbar[(long)ps * 64 + tid];
      dv[tid] = du[((long)s * EQD_HEADS + k) * 64 + tid];
    }
    __syncthreads();
    if (tid < 64) {
      double t = 0.0;
      for (int dd = 0; dd < 64; ++dd) t = fma((double)wq[tid][dd], qb[dd], t);
      r[tid] = t;
    } else if (tid < 128) {
      const int e = tid - 64;
      double t = 0.0;
      for (int dd = 0; dd < 64; ++dd) t = fma((double)wk[e][dd], dv[dd], t);
      a[e] = t * 0.125;
      a_out[((long)s * EQD_HEADS + k) * 64 + e] = t * 0.125;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      gk[q] = fma(r[e0 + q] * 0.125, dv[d], gk[q]);
      gq[q] = fma(a[e0 + q], qb[d], gq[q]);
    }
  }
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    g_wkey[((long)k * 64 + e0 + q) * 64 + d] += (float)gk[q];
    g_wquery[((long)k * 64 + e0 + q) * 64 + d] += (float)gq[q];
  }
}

// dqbar[p][d'] = sum_k sum_e W_Q,k[e][d'] a[partner(p)][k][e]      (CTA per segment p, 64 threads)
__global__ void head_dqbar_kernel(int n_pairs, eqd_head_params hp, const double* __restrict__ a, double* __restrict__ dqbar) {
  const int p = blockIdx.x, dq = threadIdx.x;
  const int s = p < n_pairs ? p + n_pairs : p - n_pairs;     // the segment whose keypoints used qbar_p
  double t = 0.0;
  for (int k = 0; k < EQD_HEADS; ++k) {
    const double* ak = a + ((long)s * EQD_HEADS + k) * 64;
    const float* w = hp.w_query + (long)k * 4096;
    for (int e = 0; e < 64; ++e) t = fma((double)w[e * 64 + dq], ak[e], t);
  }
  dqbar[(long)p * 64 + dq] = t;
}

// warp per node: pre = W_m h + b_m; dpre = dqbar[seg] / n_seg * lrelu'(pre) (* the site-3 dropout multiplier) -> dpre_out
// (D operand of dW_m); dh[n] += W_m^T dpre
template <bool DROPOUT>
__global__ void head_mean_bwd_kernel(eqd_graph g, eqd_head_params hp, const int* __restrict__ node_seg,
                                     const float* __restrict__ h, const double* __restrict__ dqbar,
                                     float* __restrict__ dpre_out, float* __restrict__ dh, DropoutArgs drop) {
  __shared__ float hs[8][64], dp[8][64];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x * 8 + w;
  if (n >= g.n_nodes) return;
  const int s = node_seg[n];
  const float inv_n = 1.f / (float)(g.seg_ptr[s + 1] - g.seg_ptr[s]);
  hs[w][lane] = h[(long)n * 64 + lane];
  hs[w][lane + 32] = h[(long)n * 64 + lane + 32];
  __syncwarp();
  float p0 = hp.b_mean[lane], p1 = hp.b_mean[lane + 32];
  for (int d = 0; d < 64; ++d) {       // w_mean is k-major [in d][out c]
    p0 = fmaf(hs[w][d], hp.w_mean[d * 64 + lane], p0);
    p1 = fmaf(hs[w][d], hp.w_mean[d * 64 + lane + 32], p1);
  }
  float g0 = (float)dqbar[(long)s * 64 + lane] * inv_n * (p0 > 0.f ? 1.f : hp.leaky_slope);
  float g1 = (float)dqbar[(long)s * 64 + lane + 32] * inv_n * (p1 > 0.f ? 1.f : hp.leaky_slope);
  if (DROPOUT) {   // columns lane and lane + 32: words lane % 4 of counters lane / 4 and 8 + lane / 4
    const unsigned long long key = dropout_key(drop);
    g0 *= dropout_mul(dropout_keep4(drop, key, lane >> 2, (unsigned)n, drop.c2), lane & 3, drop.scale);
    g1 *= dropout_mul(dropout_keep4(drop, key, 8 + (lane >> 2), (unsigned)n, drop.c2), lane & 3, drop.scale);
  }
  dpre_out[(long)n * 64 + lane] = g0;
  dpre_out[(long)n * 64 + lane + 32] = g1;
  dp[w][lane] = g0;
  dp[w][lane + 32] = g1;
  __syncwarp();
  float a0 = 0.f, a1 = 0.f;
  for (int c = 0; c < 64; ++c) {       // dh[d] = sum_c W_m[c][d] dpre[c] = sum_c w_mean[d][c] dpre[c]
    a0 = fmaf(hp.w_mean[lane * 64 + c], dp[w][c], a0);
    a1 = fmaf(hp.w_mean[(lane + 32) * 64 + c], dp[w][c], a1);
  }
  dh[(long)n * 64 + lane] += a0;
  dh[(long)n * 64 + lane + 32] += a1;
}

__global__ void node_seg_kernel(eqd_graph g, int* __restrict__ node_seg) {
  const int s = blockIdx.x;
  for (int i = g.seg_ptr[s] + threadIdx.x; i < g.seg_ptr[s + 1]; i += blockDim.x) node_seg[i] = s;
}

}  // namespace eqd

extern "C" size_t eqd_bwd_head_workspace_bytes(int32_t n_nodes, int32_t n_node_tiles, int32_t n_pairs) {
  const size_t N = n_nodes > 0 ? n_nodes : 1, B = n_pairs > 0 ? n_pairs : 1;
  return eqd_workspace_bytes(n_nodes, n_node_tiles, n_pairs)      // forward intermediates (qbar, u) are recomputed
         + eqd_align256(2 * B * EQD_HEADS * 3 * 8) * 2 + eqd_align256(B * 9 * 8) + eqd_align256(2 * B * 3 * 8)   // keypts, dY, cov, ymean
         + eqd_align256(N * 4) + eqd_align256(N * EQD_HEADS * 8) + eqd_align256(2 * B * EQD_HEADS * 3 * 8)       // node_seg, logits, stats
         + eqd_align256(2 * B * EQD_HEADS * 64 * 8) * 2 + eqd_align256(2 * B * 64 * 8);                           // du, a, dqbar
}

// Backward of eqd_keypoints + eqd_kabsch_apply.  Inputs: last-layer h (fp32) / x (fp64), `cov` as left by the forward
// (incl. any guard perturbation), the upstream gradients dcoors [N_l][3] (fp32, may be NULL), dkeypts [2B][50][3] (fp64,
// may be NULL), drot [B][9], dtrans [B][3] (fp32, may be NULL).  Outputs: dh [n][64] (fp32, overwritten), dx [n][3]
// (fp64, overwritten), dpre [n][64] (the D operand of d mlp_h_mean_ROT.0.weight = dpre^T h, reduced by the caller with
// eqd_tn_gemm), and the head weight gradients accumulated into g_wkey / g_wquery (state_dict layouts [3200][64]).
namespace eqd {
static int bwd_head(const eqd_graph* g, const eqd_head_params* hp, const float* h, const double* x, const double* cov,
                    const float* x_lig_in, const float* dcoors, const double* dkeypts, const float* drot, const float* dtrans,
                    void* workspace, size_t workspace_bytes, float* dh, double* dx, float* dpre, float* g_wkey,
                    float* g_wquery, const DropoutArgs* drop, void* stream) {
  if (!g || !hp || !h || !x || !cov || !x_lig_in || !workspace || !dh || !dx || !dpre || !g_wkey || !g_wquery)
    return EQD_ERR_BAD_ARG;
  if (workspace_bytes < eqd_bwd_head_workspace_bytes(g->n_nodes, g->n_node_tiles, g->n_pairs)) return EQD_ERR_WORKSPACE;
  if (g->n_pairs <= 0) return EQD_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t N = g->n_nodes, B = g->n_pairs;
  unsigned char* w = reinterpret_cast<unsigned char*>(workspace);
  size_t o = 0;
  auto take = [&](size_t bytes) { unsigned char* p = w + o; o += eqd_align256(bytes); return p; };
  const size_t fwd_bytes = eqd_workspace_bytes(g->n_nodes, g->n_node_tiles, g->n_pairs);
  unsigned char* fwd_ws = take(fwd_bytes);
  double* keypts = reinterpret_cast<double*>(take(2 * B * EQD_HEADS * 3 * 8));
  double* dY = reinterpret_cast<double*>(take(2 * B * EQD_HEADS * 3 * 8));
  double* cov_scratch = reinterpret_cast<double*>(take(B * 9 * 8));
  double* ymean = reinterpret_cast<double*>(take(2 * B * 3 * 8));
  int* node_seg = reinterpret_cast<int*>(take(N * 4));
  double* logits = reinterpret_cast<double*>(take(N * EQD_HEADS * 8));
  double* stats = reinterpret_cast<double*>(take(2 * B * EQD_HEADS * 3 * 8));
  double* du = reinterpret_cast<double*>(take(2 * B * EQD_HEADS * 64 * 8));
  double* a = reinterpret_cast<double*>(take(2 * B * EQD_HEADS * 64 * 8));
  double* dqbar = reinterpret_cast<double*>(take(2 * B * 64 * 8));
  // recompute qbar, u, keypoints and their means (cov_scratch is discarded: the caller's cov may carry the guard's noise)
  int rc = keypoints(g, hp, h, x, fwd_ws, fwd_bytes, keypts, ymean, cov_scratch, drop, stream);
  if (rc) return rc;
  const double* qbar = reinterpret_cast<const double*>(fwd_ws + ws_part_bytes(g->n_node_tiles) + ws_tile_ptr_bytes(g->n_pairs));
  const double* u = reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(qbar) + ws_qbar_bytes(g->n_pairs));
  eqd::kabsch_bwd_kernel<<<g->n_pairs, 128, 0, st>>>(*g, cov, ymean, keypts, x_lig_in, dcoors, dkeypts, drot, dtrans, dY);
  EQD_CUDA_LAUNCH_CHECK();
  eqd::node_seg_kernel<<<2 * g->n_pairs, 128, 0, st>>>(*g, node_seg);
  EQD_CUDA_LAUNCH_CHECK();
  eqd::kp_logits_kernel<<<(unsigned)((N * 32 + 255) / 256), 256, 0, st>>>(*g, node_seg, h, u, logits);
  EQD_CUDA_LAUNCH_CHECK();
  eqd::kp_stats_kernel<<<2 * g->n_pairs, 64, 0, st>>>(*g, logits, keypts, dY, stats);
  EQD_CUDA_LAUNCH_CHECK();
  eqd::kp_node_bwd_kernel<<<(unsigned)((N + 7) / 8), 256, 0, st>>>(*g, node_seg, x, u, dY, stats, logits, dx, dh);
  EQD_CUDA_LAUNCH_CHECK();
  eqd::kp_du_kernel<<<2 * g->n_pairs, 256, 0, st>>>(*g, logits, h, du);
  EQD_CUDA_LAUNCH_CHECK();
  eqd::head_weight_bwd_kernel<<<EQD_HEADS, 256, 0, st>>>(g->n_pairs, *hp, qbar, du, a, g_wkey, g_wquery);
  EQD_CUDA_LAUNCH_CHECK();
  eqd::head_dqbar_kernel<<<2 * g->n_pairs, 64, 0, st>>>(g->n_pairs, *hp, a, dqbar);
  EQD_CUDA_LAUNCH_CHECK();
  if (drop)
    eqd::head_mean_bwd_kernel<true><<<(unsigned)((N + 7) / 8), 256, 0, st>>>(*g, *hp, node_seg, h, dqbar, dpre, dh, *drop);
  else
    eqd::head_mean_bwd_kernel<false><<<(unsigned)((N + 7) / 8), 256, 0, st>>>(*g, *hp, node_seg, h, dqbar, dpre, dh,
                                                                             DropoutArgs{});
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}
}  // namespace eqd

extern "C" int eqd_bwd_head(const eqd_graph* g, const eqd_head_params* hp, const float* h, const double* x,
                            const double* cov, const float* x_lig_in, const float* dcoors, const double* dkeypts,
                            const float* drot, const float* dtrans, void* workspace, size_t workspace_bytes, float* dh,
                            double* dx, float* dpre, float* g_wkey, float* g_wquery, void* stream) {
  return eqd::bwd_head(g, hp, h, x, cov, x_lig_in, dcoors, dkeypts, drot, dtrans, workspace, workspace_bytes, dh, dx, dpre,
                       g_wkey, g_wquery, nullptr, stream);
}

extern "C" int eqd_bwd_head_dropout(const eqd_graph* g, const eqd_head_params* hp, const float* h, const double* x,
                                    const double* cov, const float* x_lig_in, const float* dcoors, const double* dkeypts,
                                    const float* drot, const float* dtrans, void* workspace, size_t workspace_bytes,
                                    float* dh, double* dx, float* dpre, float* g_wkey, float* g_wquery,
                                    const eqd_dropout* dropout, int32_t layer, void* stream) {
  eqd::DropoutArgs d;
  const int rc = eqd::dropout_args(dropout, layer, 3, &d);
  if (rc) return rc;
  return eqd::bwd_head(g, hp, h, x, cov, x_lig_in, dcoors, dkeypts, drot, dtrans, workspace, workspace_bytes, dh, dx, dpre,
                       g_wkey, g_wquery, dropout ? &d : nullptr, stream);
}

// =====================================================================================================================
// Batched RMSD meter (SURVEY 8f rank 3): Meter_Unbound_Bound.update_rmsd (src/utils/eval.py:19-42) for every pair of a
// batch in one launch -- ligand RMSD, receptor RMSD and the complex RMSD after a Kabsch superposition of the predicted
// complex on the true one (rigid_transform_Kabsch_3D, src/utils/protein_utils.py:31-64; reflection fix :56-59), reusing
// the 3x3 Jacobi SVD of the docking head.  One CTA per pair, fp64, fixed-order reductions.
// =====================================================================================================================
namespace eqd {

__device__ __forceinline__ void block_sum_vec(double* v, int n, double (*sh)[12], int tid) {
  __syncthreads();
  for (int q = 0; q < n; ++q) sh[tid][q] = v[q];
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1) {
    if (tid < s)
      for (int q = 0; q < n; ++q) sh[tid][q] += sh[tid + s][q];
    __syncthreads();
  }
  for (int q = 0; q < n; ++q) v[q] = sh[0][q];
  __syncthreads();
}

__global__ void __launch_bounds__(128)
rmsd_meter_kernel(eqd_graph g, const float* __restrict__ lig_pred, const float* __restrict__ rec_pred,
                  const float* __restrict__ lig_true, const float* __restrict__ rec_true, double* __restrict__ out /*[B][3]*/) {
  __shared__ double sh[128][12];
  __shared__ double Rm[9];
  const int b = blockIdx.x, B = g.n_pairs, tid = threadIdx.x;
  const int l0 = g.seg_ptr[b], l1 = g.seg_ptr[b + 1];
  const int r0 = g.seg_ptr[B + b] - g.n_lig_nodes, r1 = g.seg_ptr[B + b + 1] - g.n_lig_nodes;
  const int nl = l1 - l0, nr = r1 - r0, n = nl + nr;
  auto P = [&](int i, int c) -> double { return i < nl ? (double)lig_pred[(long)(l0 + i) * 3 + c] : (double)rec_pred[(long)(r0 + i - nl) * 3 + c]; };
  auto Q = [&](int i, int c) -> double { return i < nl ? (double)lig_true[(long)(l0 + i) * 3 + c] : (double)rec_true[(long)(r0 + i - nl) * 3 + c]; };
  double a[12];
  for (int q = 0; q < 12; ++q) a[q] = 0.0;
  for (int i = tid; i < n; i += 128) {
    double d2 = 0.0;
    for (int c = 0; c < 3; ++c) {
      const double p = P(i, c), q = Q(i, c);
      a[c] += p;
      a[3 + c] += q;
      d2 += (p - q) * (p - q);
    }
    if (i < nl) a[6] += d2; else a[7] += d2;
  }
  block_sum_vec(a, 8, sh, tid);
  const double cp[3] = {a[0] / n, a[1] / n, a[2] / n}, cq[3] = {a[3] / n, a[4] / n, a[5] / n};
  const double lig_rmsd = sqrt(a[6] / (nl > 0 ? nl : 1)), rec_rmsd = sqrt(a[7] / (nr > 0 ? nr : 1));
  double h[12];
  for (int q = 0; q < 12; ++q) h[q] = 0.0;
  for (int i = tid; i < n; i += 128)
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) h[r * 3 + c] += (P(i, r) - cp[r]) * (Q(i, c) - cq[c]);     // H = Am Bm^T (:48)
  block_sum_vec(h, 9, sh, tid);
  if (tid == 0) {
    double A[9], U[9], S[3], V[9];
    for (int q = 0; q < 9; ++q) A[q] = h[q];
    svd3(A, U, S, V);
    double R[9];
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) R[r * 3 + c] = V[r * 3] * U[c * 3] + V[r * 3 + 1] * U[c * 3 + 1] + V[r * 3 + 2] * U[c * 3 + 2];   // Vt.T @ U.T
    const double det = R[0] * (R[4] * R[8] - R[5] * R[7]) - R[1] * (R[3] * R[8] - R[5] * R[6]) + R[2] * (R[3] * R[7] - R[4] * R[6]);
    if (det < 0.0)
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[r * 3 + c] = V[r * 3] * U[c * 3] + V[r * 3 + 1] * U[c * 3 + 1] - V[r * 3 + 2] * U[c * 3 + 2];
    for (int q = 0; q < 9; ++q) Rm[q] = R[q];
  }
  __syncthreads();
  double e[12];
  for (int q = 0; q < 12; ++q) e[q] = 0.0;
  for (int i = tid; i < n; i += 128) {
    const double px = P(i, 0) - cp[0], py = P(i, 1) - cp[1], pz = P(i, 2) - cp[2];
    for (int r = 0; r < 3; ++r) {
      const double v = Rm[r * 3] * px + Rm[r * 3 + 1] * py + Rm[r * 3 + 2] * pz + cq[r] - Q(i, r);   // R p + t, t = -R cA + cB
      e[0] += v * v;
    }
  }
  block_sum_vec(e, 1, sh, tid);
  if (tid == 0) {
    out[(long)b * 3 + 0] = sqrt(e[0] / (n > 0 ? n : 1));
    out[(long)b * 3 + 1] = lig_rmsd;
    out[(long)b * 3 + 2] = rec_rmsd;
  }
}

}  // namespace eqd

// out[b] = {complex_rmsd, ligand_rmsd, receptor_rmsd} of pair b.  Coordinates are fp32 [N_l][3] / [N_r][3] in batch order
// (receptor arrays indexed by receptor-local node id).
extern "C" int eqd_rmsd_meter(const eqd_graph* g, const float* lig_pred, const float* rec_pred, const float* lig_true,
                              const float* rec_true, double* out, void* stream) {
  if (!g || !lig_pred || !rec_pred || !lig_true || !rec_true || !out) return EQD_ERR_BAD_ARG;
  if (g->n_pairs <= 0) return EQD_OK;
  eqd::rmsd_meter_kernel<<<g->n_pairs, 128, 0, (cudaStream_t)stream>>>(*g, lig_pred, rec_pred, lig_true, rec_true, out);
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}
