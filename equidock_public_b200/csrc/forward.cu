// The whole hot path behind ONE C call: IEGMN.forward + the rigid transform of Rigid_Body_Docking_Net.forward
// (rigid_docking_model.py:452-600, 657-665).  Host code only: it carves the caller's workspace and chains the
// per-stage entry points of this library on one stream, so a binding pays one foreign call (and ~40 kernel launches)
// per batch instead of ~45 calls plus as many device allocations.
#include <cstdint>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "dropout.cuh"

namespace {

inline size_t al256(size_t v) { return (v + 255) & ~(size_t)255; }

struct Carve {
  size_t h0, x0, xa, xb, ha, hb, pa, pb, aggr, mu, kv, x5, head, keypts, ymean, cov, total;
  size_t kv_bytes, x5_rows, head_bytes;
};

Carve carve(const eqd_graph* g) {
  Carve c;
  const size_t N = (size_t)(g->n_nodes > 0 ? g->n_nodes : 0), B = (size_t)(g->n_pairs > 0 ? g->n_pairs : 0);
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += al256(bytes); return at; };
  c.h0 = take(N * EQD_H0_PAD * 4);
  c.x0 = take(N * 3 * 8);
  c.xa = take(N * 3 * 8);
  c.xb = take(N * 3 * 8);
  c.ha = take(N * EQD_HID * 4);
  c.hb = take(N * EQD_HID * 4);
  c.pa = take(N * (128 + 3 * EQD_H0_PAD) * 4);
  c.pb = take(N * (128 + 3 * EQD_H0_PAD) * 4);
  c.aggr = take(N * EQD_HID * 4);
  c.mu = take(N * EQD_H0_PAD * 4);
  c.kv_bytes = eqd_kv_blocks_bytes(g->n_nodes);
  c.kv = take(c.kv_bytes);
  c.x5_rows = ((N + 7) / 8 + 8) * 8;
  c.x5 = take(c.x5_rows * 16 * 4);
  c.head_bytes = eqd_workspace_bytes(g->n_nodes, g->n_node_tiles, g->n_pairs);
  c.head = take(c.head_bytes);
  c.keypts = take(2 * B * EQD_HEADS * 3 * 8);
  c.ymean = take(2 * B * 3 * 8);
  c.cov = take(B * 9 * 8);
  c.total = o;
  return c;
}

}  // namespace

extern "C" size_t eqd_forward_workspace_bytes(const eqd_graph* g) { return g ? carve(g).total : 0; }

// ---- training stash: the per-layer inputs the backward kernels recompute from -----------------------------------------
namespace {
struct Stash {
  size_t h0, x, h, aggr, mu, total, x_stride, h_stride, a_stride, m_stride;
};
Stash stash_layout(const eqd_graph* g, int n_layers) {
  Stash s;
  const size_t N = (size_t)(g->n_nodes > 0 ? g->n_nodes : 0), L = (size_t)(n_layers > 0 ? n_layers : 0);
  s.x_stride = al256(N * 3 * 8);
  s.h_stride = al256(N * EQD_HID * 4);
  s.a_stride = al256(N * EQD_HID * 4);
  s.m_stride = al256(N * EQD_H0_PAD * 4);
  size_t o = 0;
  s.h0 = o; o += al256(N * EQD_H0_PAD * 4);
  s.x = o; o += L * s.x_stride;          // x[l] = coordinates entering layer l (x[0] = input coordinates)
  s.h = o; o += L * s.h_stride;          // h[l] = features entering layer l, l >= 1 (slot 0 unused: layer 0 reads h0)
  s.aggr = o; o += L * s.a_stride;       // aggr[l] = mean edge message of layer l
  s.mu = o; o += L * s.m_stride;         // mu[l] = attention output of layer l (row stride 72 for layer 0, else 64)
  s.total = o;
  return s;
}
}  // namespace

extern "C" size_t eqd_forward_stash_bytes(const eqd_graph* g, int32_t n_layers) { return g ? stash_layout(g, n_layers).total : 0; }
extern "C" int eqd_forward_stash_offsets(const eqd_graph* g, int32_t n_layers, size_t* out /*[9]*/) {
  if (!g || !out) return EQD_ERR_BAD_ARG;
  const Stash s = stash_layout(g, n_layers);
  out[0] = s.h0; out[1] = s.x; out[2] = s.x_stride; out[3] = s.h; out[4] = s.h_stride; out[5] = s.aggr; out[6] = s.a_stride;
  out[7] = s.mu; out[8] = s.m_stride;
  return EQD_OK;
}

extern "C" int eqd_iegmn_forward(const eqd_graph* g, const eqd_layer* const* layers, int32_t n_layers,
                                 const eqd_head_params* hp, const eqd_forward_io* io, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  return eqd_iegmn_forward_dropout(g, layers, n_layers, hp, io, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int eqd_iegmn_forward_dropout(const eqd_graph* g, const eqd_layer* const* layers, int32_t n_layers,
                                         const eqd_head_params* hp, const eqd_forward_io* io, const eqd_dropout* dropout,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  if (!g || !layers || n_layers < 1 || !hp || !io || !workspace) return EQD_ERR_BAD_ARG;
  // per-site kernel arguments: drop[li][0] = the edge stage's (sites 0, 1), drop[li][1] = node_mlp's (site 2); head: site 3
  eqd::DropoutArgs dhead{};
  if (int rc = eqd::dropout_args(dropout, n_layers, 3, &dhead)) return rc;
  if (dropout && io->layer0_fp32) return EQD_ERR_UNSUPPORTED;   // the fp32 CUDA-core twins have no dropout
  if (!io->emb || !io->res_lig || !io->res_rec || !io->mu_lig || !io->mu_rec || !io->x_lig || !io->x_rec || !io->rot ||
      !io->trans || !io->ligand_out || !io->sing || !io->status || !io->h_out || !io->x_out)
    return EQD_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(io->h_out) | reinterpret_cast<uintptr_t>(io->x_out)) & 15)
    return EQD_ERR_BAD_ARG;   // rows are written 16 bytes at a time
  for (int li = 0; li < n_layers; ++li)
    if (!layers[li]) return EQD_ERR_BAD_ARG;
  const Carve c = carve(g);
  if (workspace_bytes < c.total) return EQD_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return EQD_ERR_BAD_ARG;
  if (g->n_pairs <= 0 || g->n_nodes <= 0) return EQD_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // debugging knobs (bit mask): 1 skip the head, 2 skip the memsets, 4 synchronise after every stage, 8 stop after layer 0
  static const int dbg = getenv("EQD_FORWARD_DEBUG") ? atoi(getenv("EQD_FORWARD_DEBUG")) : 0;
  unsigned char* w = reinterpret_cast<unsigned char*>(workspace);
  float* h0 = reinterpret_cast<float*>(w + c.h0);
  double* x0 = reinterpret_cast<double*>(w + c.x0);
  double* xbuf[2] = {reinterpret_cast<double*>(w + c.xa), reinterpret_cast<double*>(w + c.xb)};
  float* hbuf[2] = {reinterpret_cast<float*>(w + c.ha), reinterpret_cast<float*>(w + c.hb)};
  float* pa = reinterpret_cast<float*>(w + c.pa);
  float* pb = reinterpret_cast<float*>(w + c.pb);
  float* aggr = reinterpret_cast<float*>(w + c.aggr);
  float* mu = reinterpret_cast<float*>(w + c.mu);
  unsigned char* kv = w + c.kv;
  float* x5 = reinterpret_cast<float*>(w + c.x5);
  double* keypts = io->keypts ? io->keypts : reinterpret_cast<double*>(w + c.keypts);
  double* ymean = io->ymean ? io->ymean : reinterpret_cast<double*>(w + c.ymean);
  double* cov = io->cov ? io->cov : reinterpret_cast<double*>(w + c.cov);
  const int N = g->n_nodes, B = g->n_pairs;
  // training: every layer's inputs (h, x), mean edge message and attention output go to the caller's stash instead of the
  // ping-pong buffers, so that the backward kernels can recompute each layer from them
  unsigned char* sb = reinterpret_cast<unsigned char*>(io->train_stash);
  Stash sl;
  if (sb) {
    sl = stash_layout(g, n_layers);
    if (io->train_stash_bytes < sl.total || (reinterpret_cast<uintptr_t>(sb) & 255)) return EQD_ERR_WORKSPACE;
    h0 = reinterpret_cast<float*>(sb + sl.h0);
    x0 = reinterpret_cast<double*>(sb + sl.x);
  }

  // rows the kernels never write but the tensor cores / TMA read: the tail of the last 8-node block and the 8 pad
  // blocks of each (K|V, split) plane, and the pad rows of x5 (they reach P.V as 0 x value: must be finite)
  if (!(dbg & 2)) {
    const size_t plane = c.kv_bytes / 6, from = (size_t)(N / 8) * 1024;
    cudaError_t me = cudaSuccess;
    for (int pl = 0; pl < 6 && me == cudaSuccess; ++pl) me = cudaMemsetAsync(kv + pl * plane + from, 0, plane - from, st);
    if (me == cudaSuccess) me = cudaMemsetAsync(x5 + (size_t)N * 16, 0, (c.x5_rows - (size_t)N) * 16 * 4, st);
    if (me == cudaSuccess) me = cudaMemsetAsync(io->status, 0, (size_t)(B + 1) * sizeof(int32_t), st);
    if (me != cudaSuccess) return -(1000 + (int)me);
  }
  auto stage_event = [&](int li, int which) {   // which: 0 edge begin, 1 edge end, 2 node begin, 3 node end
    if (io->stage_events && io->stage_events[li * 4 + which]) cudaEventRecord((cudaEvent_t)io->stage_events[li * 4 + which], st);
  };
  int rc = eqd_embed_checked(g, io->emb, io->res_lig, io->res_rec, io->mu_lig, io->mu_rec, io->x_lig, io->x_rec, h0, x0,
                             io->status, stream);
  if (rc) return rc;
  const eqd_layer* l0_l = layers[0];
  const eqd_layer_params* l0 = &l0_l->dev;
  const bool tc0 = l0->dh == EQD_H0 && l0->w_proj_tc && l0->w_node_tc && !io->layer0_fp32;
  if (tc0) rc = eqd_project_tc0(g, l0_l, h0, pa, kv, x5, stream);
  else rc = eqd_project(g, l0_l, h0, l0->dh == EQD_H0 ? EQD_H0_PAD : EQD_HID, pa, stream);
  if (rc) return rc;
  const float* h_in = h0;
  int ldh = l0->dh == EQD_H0 ? EQD_H0_PAD : EQD_HID;
  const double* x_in = x0;
  for (int li = 0; li < n_layers; ++li) {
    const eqd_layer* lp_l = layers[li];
    const eqd_layer* lpn_l = li + 1 < n_layers ? layers[li + 1] : nullptr;
    const eqd_layer_params* lp = &lp_l->dev;
    const eqd_layer_params* lpn = lpn_l ? &lpn_l->dev : nullptr;
    const bool last = lpn == nullptr;
    float* h_out = last ? io->h_out : hbuf[li & 1];
    double* x_out = last ? io->x_out : xbuf[li & 1];
    if (sb) {
      if (!last) {
        h_out = reinterpret_cast<float*>(sb + sl.h + (size_t)(li + 1) * sl.h_stride);
        x_out = reinterpret_cast<double*>(sb + sl.x + (size_t)(li + 1) * sl.x_stride);
      }
      aggr = reinterpret_cast<float*>(sb + sl.aggr + (size_t)li * sl.a_stride);
      mu = reinterpret_cast<float*>(sb + sl.mu + (size_t)li * sl.m_stride);
    }
    eqd::DropoutArgs de{}, dn{};
    if (dropout) {
      eqd::dropout_args(dropout, li, 0, &de);
      eqd::dropout_args(dropout, li, 2, &dn);
    }
    stage_event(li, 0);
    rc = eqd::edge_stage_tc(g, lp_l, pa, x_in, x0, aggr, x_out, io->status, dropout ? &de : nullptr, stream);
    if (rc) return rc;
    stage_event(li, 1);
    stage_event(li, 2);
    if (lp->dh == EQD_HID && lp->w_node_tc && (!lpn || lpn->w_proj_tc)) {
      rc = eqd::node_stage_tc(g, lp_l, lpn_l, h_in, h0, pa, aggr, kv, mu, h_out, pb, dropout ? &dn : nullptr, stream);
    } else if (li == 0 && tc0 && (!lpn || lpn->w_proj_tc)) {
      rc = eqd::node_stage_tc0(g, lp_l, lpn_l, h0, pa, aggr, kv, x5, mu, h_out, pb, dropout ? &dn : nullptr, stream);
    } else if (dropout) {
      return EQD_ERR_UNSUPPORTED;
    } else {   // fp32 CUDA-core node stage (fused projections); the next layer's tensor-core attention needs K/V blocks
      rc = eqd_node_stage(g, lp_l, lpn_l, h_in, ldh, h0, pa, aggr, h_out, pb, stream);
      if (!rc && lpn && lpn->dh == EQD_HID && lpn->w_node_tc) rc = eqd_kv_blocks(g, pb, 320, 192, 256, kv, stream);
    }
    if (rc) return rc;
    stage_event(li, 3);
    if (dbg & 4) cudaStreamSynchronize(st);
    if ((dbg & 8) && li == 0) return EQD_OK;
    float* t = pa; pa = pb; pb = t;
    h_in = h_out;
    ldh = EQD_HID;
    x_in = x_out;
  }
  if (dbg & 1) return EQD_OK;
  rc = eqd::keypoints(g, hp, h_in, x_in, w + c.head, c.head_bytes, keypts, ymean, cov, dropout ? &dhead : nullptr, stream);
  if (rc) return rc;
  return eqd_kabsch_apply(g, cov, ymean, io->x_lig, nullptr, io->rot, io->trans, io->ligand_out, io->sing, io->status, stream);
}

// ---- dropout keep masks for tests and oracles (dropout.cuh) --------------------------------------------------------------
namespace eqd {
__global__ void dropout_mask_kernel(DropoutArgs d, int rows, int cols, unsigned char* __restrict__ keep) {
  const int nc4 = (cols + 3) / 4;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)rows * nc4) return;
  const int r = (int)(i / nc4), c4 = (int)(i - (long)r * nc4);
  const unsigned bits = dropout_keep4(d, dropout_key(d), (unsigned)c4, (unsigned)r, d.c2);
  for (int j = 0; j < 4 && c4 * 4 + j < cols; ++j) keep[(long)r * cols + c4 * 4 + j] = (bits >> j) & 1u;
}
}  // namespace eqd

extern "C" int eqd_dropout_mask(const eqd_dropout* dropout, int32_t layer, int32_t site, int32_t rows, int32_t cols,
                                uint8_t* keep, void* stream) {
  if (!dropout || !keep || rows < 0 || cols < 0) return EQD_ERR_BAD_ARG;
  eqd::DropoutArgs d{};
  if (int rc = eqd::dropout_args(dropout, layer, site, &d)) return rc;
  const long n = (long)rows * ((cols + 3) / 4);
  if (n == 0) return EQD_OK;
  eqd::dropout_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d, rows, cols, keep);
  EQD_CUDA_LAUNCH_CHECK();
  return EQD_OK;
}

// Thin CUDA event helpers so that a binding without its own CUDA runtime access can time the stages of
// eqd_iegmn_forward (io->stage_events) on the launching stream.
extern "C" void* eqd_event_create(void) {
  cudaEvent_t e = nullptr;
  return cudaEventCreate(&e) == cudaSuccess ? (void*)e : nullptr;
}
extern "C" void eqd_event_destroy(void* e) {
  if (e) cudaEventDestroy((cudaEvent_t)e);
}
extern "C" float eqd_event_elapsed_ms(void* a, void* b) {
  float ms = -1.f;
  if (!a || !b || cudaEventElapsedTime(&ms, (cudaEvent_t)a, (cudaEvent_t)b) != cudaSuccess) return -1.f;
  return ms;
}
