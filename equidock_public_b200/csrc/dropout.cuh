// Counter-based dropout masks (training with args['dropout'] > 0; the four nn.Dropout sites of rigid_docking_model.py
// :119-159, 427-438).  Stateless: the mask of an element is a pure function of (key, layer, site, row, column, rank), so
// the backward kernels regenerate the forward's mask instead of storing it.
//
//   Philox4x32-10 (Salmon et al., SC'11; Random123 constants), key = the 64-bit per-forward key {lo, hi},
//   counter = {column / 4, row, 4 * layer + site, rank};  word j of the result belongs to column 4 * (column / 4) + j;
//   keep iff word >= threshold (threshold = min(round(p 2^32), 2^32 - 1)); a kept element is scaled by fp32(1 / (1 - p)).
// Sites: 0 edge_mlp (z1, edge rows), 1 coors_mlp (z3, edge rows), 2 node_mlp (u5, node rows), 3 mlp_h_mean_ROT (node rows,
// layer = n_layers).  Rows are global edge ids in CSR order (sites 0, 1) or global node ids (sites 2, 3).
// Restated in numpy in tests/dropout_oracle.py.
#pragma once
#include <stdint.h>

#include "../../include/eqd_iegmn.h"

namespace eqd {

// What a kernel receives by value: the key pointer (device memory, read at use) and the mask constants.  c2 = 4*layer+site
// of the first site the kernel masks (a kernel with two sites uses c2 and c2 + 1).
struct DropoutArgs {
  const unsigned long long* key;
  unsigned thr;
  float scale;
  unsigned rank;
  unsigned c2;
};

// Host: validates an eqd_dropout descriptor and fills the kernel arguments of (layer, site).  NULL = no dropout (EQD_OK,
// `out` untouched).
inline int dropout_args(const eqd_dropout* d, int layer, int site, DropoutArgs* out) {
  if (!d) return EQD_OK;
  if (!d->key || layer < 0 || site < 0 || site > 3 || !(d->scale >= 1.f && d->scale < 3.0e38f)) return EQD_ERR_BAD_ARG;
  out->key = reinterpret_cast<const unsigned long long*>(d->key);
  out->thr = d->threshold;
  out->scale = d->scale;
  out->rank = d->rank;
  out->c2 = 4u * (unsigned)layer + (unsigned)site;
  return EQD_OK;
}

// Stage entry points with a dropout argument (NULL = the inference kernels); the exported eqd_* functions wrap them.
int edge_stage_tc(const eqd_graph* g, const eqd_layer* p_l, const float* proj, const double* x_in, const double* x_orig,
                  float* aggr, double* x_out, int32_t* status, const DropoutArgs* drop, void* stream);
int node_stage_tc(const eqd_graph* g, const eqd_layer* p_l, const eqd_layer* p_next_l, const float* h_in, const float* h0,
                  const float* proj, const float* aggr, void* kv, float* mu, float* h_out, float* proj_next,
                  const DropoutArgs* drop, void* stream);
int node_stage_tc0(const eqd_graph* g, const eqd_layer* p_l, const eqd_layer* p_next_l, const float* h0, const float* proj,
                   const float* aggr, void* kv, const float* x5, float* mu, float* h_out, float* proj_next,
                   const DropoutArgs* drop, void* stream);
int keypoints(const eqd_graph* g, const eqd_head_params* hp, const float* h, const double* x, void* workspace,
              size_t workspace_bytes, double* keypts, double* ymean, double* cov, const DropoutArgs* drop, void* stream);

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, unsigned k0, unsigned k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
  }
  return c;
}

// Keep bits of 4 consecutive columns [4 c0, 4 c0 + 4) of one row: bit j <-> column 4 c0 + j.
__device__ __forceinline__ unsigned dropout_keep4(const DropoutArgs& d, unsigned long long key, unsigned c0, unsigned row,
                                                  unsigned c2) {
  const uint4 w = philox4x32_10(make_uint4(c0, row, c2, d.rank), (unsigned)key, (unsigned)(key >> 32));
  return (unsigned)(w.x >= d.thr) | ((unsigned)(w.y >= d.thr) << 1) | ((unsigned)(w.z >= d.thr) << 2) |
         ((unsigned)(w.w >= d.thr) << 3);
}

// Keep bits of 32 consecutive columns [4 c0, 4 c0 + 32): 8 Philox calls, bit j <-> column 4 c0 + j.
__device__ __forceinline__ unsigned dropout_keep32(const DropoutArgs& d, unsigned long long key, unsigned c0, unsigned row,
                                                   unsigned c2) {
  unsigned bits = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) bits |= dropout_keep4(d, key, c0 + j, row, c2) << (4 * j);
  return bits;
}

__device__ __forceinline__ unsigned long long dropout_key(const DropoutArgs& d) { return __ldg(d.key); }

// Multiplier of one element: scale if kept, else 0.
__device__ __forceinline__ float dropout_mul(unsigned bits, int j, float scale) { return (bits >> j) & 1u ? scale : 0.f; }

}  // namespace eqd
