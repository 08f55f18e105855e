/*
 * eqd_iegmn.h -- C ABI of the B200 (sm_100a) IEGMN forward engine.
 *
 * Drop-in boundary for the ONE hot path of octavian-ganea/equidock_public:
 *   src/model/rigid_docking_model.py  IEGMN_Layer.forward (:189-352), IEGMN.forward (:451-602),
 *   Rigid_Body_Docking_Net.forward (:642-692).
 * The reference has no FFI of its own (pure Python over torch/DGL); these entry points are what a
 * binding for that path would call.  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - plain C: device pointers + sizes + a cudaStream_t passed as void*; no torch types.
 *   - the CALLER owns every buffer (inputs, outputs, workspace); the library never allocates,
 *     never synchronises the stream, keeps no global mutable state (thread-safe per stream).
 *   - every function returns 0 on success or a negative EQD_ERR_* code; kernel launch errors are
 *     returned as -(1000 + cudaError_t).
 *   - all matrices are row-major fp32 unless stated; coordinates inside the engine are fp64.
 *
 * Node / edge numbering of a batch of B protein pairs (mirrors dgl.batch of the reference's
 * heterograph, src/utils/train_utils.py:61-100): ligand nodes of pair 0..B-1, then receptor nodes
 * of pair 0..B-1 ("global node id").  Segment s < B is the ligand of pair s, segment B+s its
 * receptor; seg_ptr[2B+1] are global node offsets.  Edges are sorted by destination (CSR): edge e
 * = (col_src[e] -> the node whose row contains e), meaning "src is one of dst's k nearest
 * neighbours" (src/utils/protein_utils.py:339-346).
 */
#ifndef EQD_IEGMN_H
#define EQD_IEGMN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EQD_ABI_VERSION 9

#define EQD_EDGE_FEATS 27     /* input_edge_feats_dim, protein_utils.py:71-86 + :373-389 */
#define EQD_N_RBF 15          /* all_sigmas_dist = 1.5**s, rigid_docking_model.py:116 */
#define EQD_HID 64            /* iegmn_lay_hid_dim (out_feats_dim) */
#define EQD_H0 69             /* residue_emb_dim 64 + 5 surface features, :382-388 */
#define EQD_H0_PAD 72         /* row stride of padded 69-wide tensors */
#define EQD_N_RES_TYPES 21    /* nn.Embedding(21, 64), :382 */
#define EQD_HEADS 50          /* num_att_heads */
#define EQD_TILE_ROWS 128     /* rows (edges / nodes) per CTA tile */

enum {
  EQD_OK = 0,
  EQD_ERR_BAD_ARG = -1,       /* null pointer / size out of range */
  EQD_ERR_UNSUPPORTED = -2,   /* e.g. layer width other than 64 / 69, in-degree > 128 */
  EQD_ERR_WORKSPACE = -3      /* workspace smaller than eqd_workspace_bytes() */
};

/* per-pair status bits written by eqd_kabsch_apply (rigid_docking_model.py:570-584) */
#define EQD_STATUS_SVD_DEGENERATE 1  /* guard :574 fired: min S < 1e-3 or min |S_i^2-S_j^2| < 1e-2 */
#define EQD_STATUS_NAN 2             /* assert :570 would have failed */
/* global status bit (status[n_pairs]) */
#define EQD_STATUS_DEGREE_OVERFLOW 4 /* some node has more than max_in_degree in-edges */
#define EQD_STATUS_BAD_RESIDUE 8     /* a res_feat index outside [0, 21): nn.Embedding (:460) would raise IndexError */

/* ---- batch topology (all pointers device memory) ------------------------------------------ */
typedef struct eqd_graph {
  int32_t n_pairs;            /* B */
  int32_t n_nodes;            /* sum N_l + sum N_r */
  int32_t n_lig_nodes;        /* sum N_l */
  int32_t n_edges;            /* sum E_l + sum E_r */
  int32_t n_lig_edges;        /* sum E_l */
  int32_t max_in_degree;      /* upper bound on in-degree (graph_max_neighbor, 10); <= 128 */
  const int32_t* seg_ptr;     /* [2B+1] global node offsets of the 2B segments */
  const int32_t* row_ptr;     /* [n_nodes+1] CSR-by-destination edge offsets */
  const int32_t* col_src;     /* [n_edges] global source node of every edge */
  const int32_t* edge_dst;    /* [n_edges] global destination node of every edge */
  const float* he_lig;        /* [n_lig_edges][27] edges['ll'].data['he'] */
  const float* he_rec;        /* [n_edges-n_lig_edges][27] edges['rr'].data['he'] */
  int32_t n_node_tiles;       /* number of (segment, first node) tiles of <=128 nodes */
  const int32_t* node_tiles;  /* [n_node_tiles][2] = {segment, first global node} */
} eqd_graph;

/* ---- one IEGMN_Layer's parameters, repacked k-major (in-dim x out-dim) --------------------- */
/* dh = layer input width (69 for layer 0, else 64), dhp = 72 / 64 its padded width.
 * "k-major" = element [k][n] multiplies input feature k into output n, i.e. the transpose of
 * the nn.Linear weight in the reference state_dict; padded rows/cols are zero.               */
typedef struct eqd_layer_params {
  int32_t dh, dhp;
  /* node projections of h (one GEMM): column groups
   *   [0,64)            Psrc = h . edge_mlp.0.weight[:, 0:dh]^T
   *   [64,128)          Pdst = h . edge_mlp.0.weight[:, dh:2dh]^T + edge_mlp.0.bias
   *   [128,128+dhp)     Q = LeakyReLU(h . att_mlp_Q.0.weight^T)
   *   [128+dhp,+2dhp)   K = LeakyReLU(h . att_mlp_K.0.weight^T)
   *   [128+2dhp,+3dhp)  V = h . att_mlp_V.0.weight^T                                        */
  const float* w_proj;        /* [dhp][128+3*dhp] */
  const float* b_proj;        /* [128+3*dhp] */
  const float* w_edge1;       /* [44][64]: rows 0..26 he, 27..41 rbf, 42..43 zero (edge_mlp.0.weight[:, 2dh:]^T) */
  const float* edge_ln_g;     /* [64] edge_mlp.3.weight */
  const float* edge_ln_b;     /* [64] edge_mlp.3.bias */
  const float* w_edge2;       /* [64][64] edge_mlp.4.weight^T */
  const float* b_edge2;       /* [64] */
  const float* w_coor1;       /* [64][64] coors_mlp.0.weight^T */
  const float* b_coor1;       /* [64] */
  const float* w_coor2;       /* [64] coors_mlp.4.weight */
  float b_coor2;              /* coors_mlp.4.bias */
  /* tensor-core edge stage (tcgen05): the three edge-side weight matrices, each split into 3 bf16 terms
   * (w ~ w0+w1+w2, round-to-nearest) and stored in the UMMA canonical K-major no-swizzle layout
   *   element (n,k) of split s at  base + s*split_bytes + (k/8)*1024 + (n/8)*128 + (n%8)*16 + (k%8)*2
   * GEMM1 = edge_mlp.0.weight[:, 2dh:] ([64][48], K 42 -> 48, base 0, split 6144 B); GEMM2+3 = the stacked
   * [128][64] panel [edge_mlp.4.weight ; coors_mlp.0.weight @ edge_mlp.4.weight] (base 18432, split 16384 B,
   * k-chunk stride 2048 B): msg and the coordinate MLP's hidden layer are both linear in the LayerNorm output.
   * 67584 B, 16B-aligned. */
  const void* w_edge_tc;
  /* tensor-core node stage (dh == 64 layers only; NULL for the 69-wide layer 0). Same bf16x3 UMMA panels:
   *   w_node_tc : node_mlp.0.weight padded to [64][272] (K order h | aggr | mu | h0(69) | 0) at base 0, split
   *               34816 B; node_mlp.4.weight [64][64] at base 104448, split 8192 B            (129024 B)
   *   w_proj_tc : this layer's projection [Psrc|Pdst|Q|K|V] as 5 groups x 3 splits x 8192 B   (122880 B)
   * (their biases / LayerNorm vectors travel in eqd_layer_consts, below)                                 */
  const void* w_node_tc;
  const void* w_proj_tc;
  const float* w_node1;       /* [dhp+64+dhp+72][dhp] node_mlp.0.weight^T, row blocks [h | aggr_msg | mu | h0] */
  const float* b_node1;       /* [dhp] */
  const float* node_ln_g;     /* [dhp] node_mlp.3.weight (pad 0) */
  const float* node_ln_b;     /* [dhp] */
  const float* w_node2;       /* [dhp][64] node_mlp.4.weight^T */
  const float* b_node2;       /* [64] */
  float skip_weight_h;        /* args['skip_weight_h'] (applied only when dh == 64, :332-337) */
  float x_connection_init;    /* args['x_connection_init'] (:286-292) */
  float leaky_slope;          /* args['leakyrelu_neg_slope'] */
} eqd_layer_params;

/* Launch-time constants of the tensor-core kernels, BY VALUE in host memory: the launcher copies them into the kernel's
 * constant parameter space (they are operands of the epilogue FFMAs), so they never live behind a device pointer.
 *   edge      : edge_mlp.3.weight, edge_mlp.3.bias, edge_mlp.4.bias, (coors_mlp.0.weight @ edge_mlp.4.bias +
 *               coors_mlp.0.bias), coors_mlp.4.weight
 *   node      : dh == 64: [4][64] = node_mlp.0.bias, node_mlp.3.weight, node_mlp.3.bias, node_mlp.4.bias;
 *               dh == 69: [80 + 80 + 80 + 64], the first three zero padded to 80
 *   proj_bias : [320] = b_proj of the five 64-wide groups (dh == 69: only edge_mlp.0.bias at [64, 128))            */
typedef struct eqd_layer_consts {
  float edge[5][64];
  float node[304];
  float proj_bias[320];
} eqd_layer_consts;

/* One IEGMN layer as the entry points take it: a HOST-resident descriptor.  `dev` holds device pointers and scalars only
 * and is what kernels receive by value (a binding may keep or upload it wholesale); `consts` holds host VALUES.  Entry
 * points of the fp32 FFMA path and of the backward read `dev` only.                                                 */
typedef struct eqd_layer {
  eqd_layer_params dev;
  eqd_layer_consts consts;
} eqd_layer;

/* ---- keypoint read-out parameters (IEGMN.__init__ :427-438), reference layouts ------------- */
typedef struct eqd_head_params {
  const float* w_mean;        /* [64][64] mlp_h_mean_ROT.0.weight^T (k-major) */
  const float* b_mean;        /* [64] */
  const float* w_key;         /* [3200][64] att_mlp_key_ROT.0.weight, as in the state_dict */
  const float* w_query;       /* [3200][64] att_mlp_query_ROT.0.weight, as in the state_dict */
  const double* m_qk;         /* [50][64][64] fp64, written once per model by eqd_head_fold() from w_key / w_query:
                                 m_qk[k][d'][d] = sum_e w_query[64k+e][d'] w_key[64k+e][d] / 8.  Device memory, 16-byte aligned. */
  float leaky_slope;
} eqd_head_params;

int eqd_abi_version(void);

/* Bytes of scratch the layer / head entry points need for this graph (host-side arithmetic). */
size_t eqd_workspace_bytes(int32_t n_nodes, int32_t n_node_tiles, int32_t n_pairs);

/* Input stage, IEGMN.forward :452-471.
 *   h0[n][72]  = [Embedding(res_feat.long()) (64) | log(mu_r_norm) (5) | 0 0 0]
 *   x64[n][3]  = ligand new_x / receptor x, widened to fp64                                  */
int eqd_embed(const eqd_graph* g, const float* emb /*[21][64]*/,
              const float* res_feat_lig, const float* res_feat_rec,   /* [N][1] fp32-encoded ints */
              const float* mu_lig, const float* mu_rec,               /* [N][5] */
              const float* x_lig /* new_x */, const float* x_rec /* x */, /* [N][3] */
              float* h0, double* x64, void* stream);
/* Same, and ORs EQD_STATUS_BAD_RESIDUE into status[n_pairs] when a residue index is out of range (status may be NULL). */
int eqd_embed_checked(const eqd_graph* g, const float* emb, const float* res_feat_lig, const float* res_feat_rec,
                      const float* mu_lig, const float* mu_rec, const float* x_lig, const float* x_rec,
                      float* h0, double* x64, int32_t* status /* [n_pairs+1] */, void* stream);

/* Node projections for a layer (see eqd_layer_params.w_proj): proj[n][128+3*dhp]. */
int eqd_project(const eqd_graph* g, const eqd_layer* p, const float* h, int32_t ldh,
                float* proj, void* stream);

/* Edge stage of IEGMN_Layer.forward (:204-237, 263-292): RBF, edge MLP, coordinate MLP, mean
 * aggregation at the destination, coordinate update.
 *   aggr[n][64] = mean_e msg_e ;  x_out[n] = eta*x_orig[n] + (1-eta)*x_in[n] + mean_e x_rel*phi
 * Runs on tcgen05 tensor cores (bf16x3 operand split, fp32 accumulation in TMEM).  he_lig / he_rec must be
 * 16-byte aligned and readable up to the next 16-byte boundary past their end (TMA bulk copies).          */
int eqd_edge_stage(const eqd_graph* g, const eqd_layer* p, const float* proj,
                   const double* x_in, const double* x_orig, float* aggr, double* x_out,
                   int32_t* status /* [n_pairs+1] */, void* stream);

/* Same contract on the fp32 CUDA cores (FFMA); kept as the validation twin of the tensor-core kernel. */
int eqd_edge_stage_ffma(const eqd_graph* g, const eqd_layer* p, const float* proj,
                        const double* x_in, const double* x_orig, float* aggr, double* x_out,
                        int32_t* status /* [n_pairs+1] */, void* stream);

/* Node stage (:244-256, 319-349): segmented cross attention mu = softmax(q k^T) v over the partner
 * protein, node MLP + LayerNorm + skip -> h_out[n][64]; if p_next != NULL also the next layer's
 * projections (fused eqd_project on h_out) into proj_next.                                    */
int eqd_node_stage(const eqd_graph* g, const eqd_layer* p, const eqd_layer* p_next,
                   const float* h_in, int32_t ldh, const float* h0, const float* proj,
                   const float* aggr, float* h_out, float* proj_next, void* stream);

/* ---- tensor-core node stage (tcgen05, layers with dh == 64) ---------------------------------------------
 * K and V of every node travel as bf16x3 "8-node blocks": kv[which 2 (K,V)][split 3][n/8 (+8 zero pad
 * blocks)][d/8][n%8][d%8] bf16 (1 KB per block), so a run of blocks is a ready UMMA B operand for TMA.   */
size_t eqd_kv_blocks_bytes(int32_t n_nodes);
/* proj[n][320] = [Psrc|Pdst|Q|K|V](h[n]) for a dh==64 layer.  With kv != NULL, K and V are written ONLY as
 * bf16x3 blocks into kv and the fp32 columns 192..319 of proj are left untouched (nothing downstream reads them). */
int eqd_project_tc(const eqd_graph* g, const eqd_layer* p, const float* h /*[n][64]*/, float* proj,
                   void* kv, void* stream);
/* The same for the 69-wide layer 0 (h = h0 [n][72], K padded to 80): proj[n][344] gets Psrc | Pdst | Q[0:64] at
 * columns 0 / 64 / 128 (the positions the fp32 layer-0 layout uses); K[0:64], V[0:64] go to kv as bf16x3 blocks;
 * channels 64..68 of K, V, Q go to x5[n][16] = [K64..67 | V64..67 | K68 V68 | Q64..68 | 0] (fp32), which is what
 * eqd_attention_tc0 adds to the 64-wide tensor-core products.  kv and x5 are required; x5 must have
 * 8 * (ceil(n / 8) + 8) rows, the rows past n zero (attention reads whole 64-key chunks).                     */
int eqd_project_tc0(const eqd_graph* g, const eqd_layer* p, const float* h0 /*[n][72]*/, float* proj /*[n][344]*/,
                    void* kv, float* x5 /*[n][16]*/, void* stream);
/* K/V blocks from the fp32 columns of an existing projection buffer (row stride pw floats). */
int eqd_kv_blocks(const eqd_graph* g, const float* proj, int32_t pw, int32_t koff, int32_t voff, void* kv,
                  void* stream);
/* mu[n][64] = softmax_j(q_n . k_j) v_j over the partner protein (:46-64, 247-256); proj row stride 320. */
int eqd_attention_tc(const eqd_graph* g, const float* proj, const void* kv, float* mu, void* stream);
/* h_out = skip(node_mlp([h | aggr | mu | h0])) (:319-337). */
int eqd_node_mlp_tc(const eqd_graph* g, const eqd_layer* p, const float* h_in, const float* aggr,
                    const float* mu, const float* h0, float* h_out, void* stream);
/* Node stage of a dh==64 layer on the tensor cores = attention + node MLP (+ the next layer's projections and
 * K/V blocks when p_next != NULL).  kv holds this layer's K/V blocks on entry, the next layer's on exit;
 * mu is [n][64] scratch.                                                                                   */
int eqd_node_stage_tc(const eqd_graph* g, const eqd_layer* p, const eqd_layer* p_next,
                      const float* h_in, const float* h0, const float* proj, const float* aggr, void* kv,
                      float* mu, float* h_out, float* proj_next, void* stream);

/* ---- the 69-wide layer 0 on the tensor cores.  For p->dh == 69 the tensor-core panel fields of eqd_layer_params hold
 *   w_proj_tc : 5 groups [64][80] (Psrc, Pdst, Q[0:64], K[0:64], V[0:64]; K = h0 channels 69 -> 80) x 3 splits x 10240 B,
 *               then one [16][80] group (rows K64..67, V64..67, K68, V68, Q64..68, 0) x 3 splits x 2560 B    (161280 B)
 *   w_node_tc : node_mlp.0.weight with the h and h0 blocks folded (h = h0 in layer 0), [80][224] = 69 -> 80 outputs over
 *               K = [h0 80 | aggr 64 | mu 80], 3 splits x 35840 B; node_mlp.4.weight as [64][80] at 107520    (138240 B)
 *   consts.node = [80 + 80 + 80 + 64] (node_mlp.0.bias, node_mlp.3.weight, node_mlp.3.bias zero padded, node_mlp.4.bias);
 *   consts.proj_bias = [320] with edge_mlp.0.bias at [64, 128).
 * eqd_attention_tc0: mu[n][72] = softmax(q k^T) v over the partner protein with d = 69: channels 0..63 on the tensor cores
 * from proj[n][344] (Q at column 128) and kv, channels 64..68 in fp32 from x5; columns 69..71 of mu are written as 0.
 * eqd_node_mlp_tc0: h_out[n][64] = node_mlp([h0 | aggr | mu | h0]) without skip connection (:332).
 * eqd_node_stage_tc0 = attention + node MLP + (p_next != NULL) the 64-wide projections of layer 1.              */
int eqd_attention_tc0(const eqd_graph* g, const float* proj /*[n][344]*/, const void* kv, const float* x5 /*[n+72][16]*/,
                      float* mu /*[n][72]*/, void* stream);
int eqd_node_mlp_tc0(const eqd_graph* g, const eqd_layer* p, const float* h0 /*[n][72]*/, const float* aggr,
                     const float* mu /*[n][72]*/, float* h_out /*[n][64]*/, void* stream);
int eqd_node_stage_tc0(const eqd_graph* g, const eqd_layer* p, const eqd_layer* p_next, const float* h0,
                       const float* proj, const float* aggr, void* kv, const float* x5, float* mu, float* h_out,
                       float* proj_next, void* stream);

/* One whole IEGMN_Layer.forward = eqd_edge_stage + eqd_node_stage (proj must hold this layer's
 * projections on entry; holds the next layer's on exit when p_next != NULL).                  */
int eqd_iegmn_layer_forward(const eqd_graph* g, const eqd_layer* p, const eqd_layer* p_next,
                            const float* h_in, int32_t ldh, const float* h0,
                            const double* x_in, const double* x_orig,
                            float* proj, float* proj_next, float* aggr,
                            float* h_out, double* x_out, int32_t* status, void* stream);

/* Weights-only fold of the 50-head key / query projections (att_mlp_key_ROT, att_mlp_query_ROT :427-438) into
 * m_qk (see eqd_head_params), so that the per-protein logits are h_j . (m_qk[k]^T qbar) (:544-546, :555-557).
 * Call once after loading a checkpoint; eqd_keypoints() reads hp->m_qk.                                       */
int eqd_head_fold(const eqd_head_params* hp, double* m_qk /*[50][64][64]*/, void* stream);

/* Keypoint read-out (IEGMN.forward :521-567): mean-pooled queries, 50-head attention over each
 * protein's nodes, keypoints Y (fp64 [2B][50][3], segment order), their means and the 3x3
 * covariance A = (Y_rec - mean)^T (Y_lig - mean) per pair (cov[B][9], ymean[2B][3]).        */
int eqd_keypoints(const eqd_graph* g, const eqd_head_params* hp, const float* h /*[n][64]*/,
                  const double* x /*[n][3] last-layer coords*/, void* workspace, size_t workspace_bytes,
                  double* keypts, double* ymean, double* cov, void* stream);

/* Kabsch + rigid transform (:571-589, 657-665): SVD of cov, guard test, T = U diag(1,1,sign det A) V^T,
 * b = ymean_rec - T ymean_lig; ligand_out[n] = T new_x[n] + b for every ligand node.
 * Outputs fp32 (what the reference returns): rot[B][9], trans[B][3], ligand_out[n_lig][3];
 * sing[B][3] fp64 singular values; status[B] gets EQD_STATUS_* bits (caller zero-initialises).
 * pair_mask: NULL = all pairs, else only pairs with pair_mask[b] != 0 are (re)computed.       */
int eqd_kabsch_apply(const eqd_graph* g, const double* cov, const double* ymean, const float* x_lig_in,
                     const int32_t* pair_mask, float* rot, float* trans, float* ligand_out,
                     double* sing, int32_t* status, void* stream);


/* ---- the whole hot path in one call ----------------------------------------------------------------------------------
 * eqd_iegmn_forward = IEGMN.forward (rigid_docking_model.py:452-600: embedding, the n_layers IEGMN layers, keypoint
 * read-out, Kabsch) + the rigid transform of the ligand (Rigid_Body_Docking_Net.forward :657-665), chained on `stream`
 * out of the entry points above.  Nothing is allocated: the caller provides eqd_forward_workspace_bytes(g) bytes of
 * 256-byte aligned device memory.  Layers whose tensor-core panels are present run on the tensor cores, the others on
 * the fp32 CUDA-core kernels.  All pointers are device memory unless noted.                                          */
typedef struct eqd_forward_io {
  /* inputs (reference tensors: residue_emb_layer.weight; ndata['res_feat'], ['mu_r_norm'], ligand ['new_x'], receptor ['x']) */
  const float* emb;           /* [21][64] */
  const float* res_lig;       /* [N_l][1] fp32-encoded residue ids */
  const float* res_rec;
  const float* mu_lig;        /* [N_l][5] */
  const float* mu_rec;
  const float* x_lig;         /* [N_l][3] */
  const float* x_rec;
  /* outputs */
  float* rot;                 /* [B][9]  */
  float* trans;               /* [B][3]  */
  float* ligand_out;          /* [N_l][3] transformed ligand coordinates */
  double* sing;               /* [B][3] singular values */
  int32_t* status;            /* [B+1] EQD_STATUS_* bits, zeroed by the call */
  float* h_out;               /* [n][64] last layer's node features  (ndata['hv_iegmn_out']) */
  double* x_out;              /* [n][3]  last layer's coordinates    (ndata['x_iegmn_out'])  */
  double* keypts;             /* [2B][50][3] or NULL */
  double* cov;                /* [B][9] Kabsch covariances (eqd_kabsch_apply can be replayed on them) or NULL */
  double* ymean;              /* [2B][3] keypoint means (needed for such a replay) or NULL */
  /* optional: HOST array of 4*n_layers cudaEvent_t handles (edge begin, edge end, node begin, node end per layer) recorded
   * on `stream`; NULL entries are skipped.  eqd_event_create / _elapsed_ms / _destroy wrap the CUDA calls.          */
  void* const* stage_events;
  int32_t layer0_fp32;        /* != 0: keep the 69-wide layer 0 on the fp32 CUDA-core kernels */
  /* training: NULL, or eqd_forward_stash_bytes(g, n_layers) bytes of 256-byte aligned device memory that receives every
   * layer's inputs and intermediate node tensors (layout: eqd_forward_stash_offsets) for the backward entry points */
  void* train_stash;
  size_t train_stash_bytes;
} eqd_forward_io;

size_t eqd_forward_workspace_bytes(const eqd_graph* g);
size_t eqd_forward_stash_bytes(const eqd_graph* g, int32_t n_layers);
/* out[9] = byte offsets / strides inside the stash: h0 [n][72] f32 | x[l] [n][3] f64 (offset, stride per layer; x[0] = the
 * input coordinates) | h[l] [n][64] f32, l >= 1 (offset, stride) | aggr[l] [n][64] f32 (offset, stride) | mu[l] f32, row
 * stride 72 for the 69-wide layer 0 and 64 otherwise (offset, stride) */
int eqd_forward_stash_offsets(const eqd_graph* g, int32_t n_layers, size_t* out);
int eqd_iegmn_forward(const eqd_graph* g, const eqd_layer* const* layers, int32_t n_layers,
                      const eqd_head_params* hp, const eqd_forward_io* io, void* workspace, size_t workspace_bytes,
                      void* stream);

/* ---- dropout in training (the four nn.Dropout sites of rigid_docking_model.py :119-159, 427-438) --------------------------
 * Counter-based masks, so that the backward regenerates the forward's mask and nothing is stored.  Element (row, col) of
 * site s in layer l is kept iff word (col % 4) of Philox4x32-10(counter = {col / 4, row, 4 l + s, rank}, key = {*key low 32
 * bits, high 32 bits}) >= threshold; a kept element is multiplied by `scale`, a dropped one by 0.  Sites: 0 edge_mlp (after
 * its first Linear, 64 wide), 1 coors_mlp (64), 2 node_mlp (64; 69 in the 69-wide layer 0), 3 mlp_h_mean_ROT (64, layer =
 * n_layers).  Rows: global edge id in CSR order (sites 0, 1), global node id (sites 2, 3).  The mask multiplies the LeakyReLU
 * output, which equals the reference's dropout-then-LeakyReLU (LeakyReLU is positively homogeneous).
 * A NULL descriptor means no dropout: the entry points below then run exactly the kernels of the inference path.          */
typedef struct eqd_dropout {
  const uint64_t* key;        /* DEVICE memory: the 64-bit key of this forward (read by the kernels, no host sync) */
  uint32_t threshold;         /* min(round(p 2^32), 2^32 - 1) */
  float scale;                /* fp32(1 / (1 - p)) */
  uint32_t rank;              /* data-parallel rank: equally seeded ranks draw different masks */
} eqd_dropout;

/* eqd_iegmn_forward with dropout (tensor-core path only: EQD_ERR_UNSUPPORTED with io->layer0_fp32 or a layer without
 * tensor-core panels, whose fp32 CUDA-core twins have no dropout). */
int eqd_iegmn_forward_dropout(const eqd_graph* g, const eqd_layer* const* layers, int32_t n_layers,
                              const eqd_head_params* hp, const eqd_forward_io* io, const eqd_dropout* dropout,
                              void* workspace, size_t workspace_bytes, void* stream);
/* keep[r][c] = 1 / 0 for rows 0..rows-1, columns 0..cols-1 of (layer, site) (device memory; for tests and oracles). */
int eqd_dropout_mask(const eqd_dropout* dropout, int32_t layer, int32_t site, int32_t rows, int32_t cols, uint8_t* keep,
                     void* stream);

/* =====================================================================================================================
 * BACKWARD of the path (training: BASELINE configs 3-4).  The reference has no backward code: these entry points are
 * what a binding would call from torch.autograd.Function.backward in place of `loss.backward()` (src/train.py:154)
 * walking rigid_docking_model.py in reverse.  Same conventions as above (device pointers, caller-owned buffers, stream).
 * Flow for one batch: eqd_iegmn_forward with io->train_stash set -> (losses) -> eqd_bwd_head -> for every layer, last to
 * first: eqd_project (recompute this layer's Psrc|Pdst|Q|K|V in fp32) -> eqd_bwd_node_mlp -> eqd_bwd_attention ->
 * eqd_bwd_edge -> eqd_bwd_edge_gather -> eqd_bwd_project, each followed by eqd_tn_gemm + eqd_grad_reduce for its weight
 * gradients -> eqd_bwd_embed.  All reductions run in a fixed order: gradients are bit-reproducible for a given batch.
 * ================================================================================================================== */

/* Generic weight-gradient reduction  partial[c][k][n] = alpha * sum_{rows of chunk c} X[row][k] * D[row][n]  (and, if
 * colsum != NULL, colsum[c][n] = alpha * sum D[row][n]: the bias gradient).  K, ncols, ldx, ldd multiples of 4; X and D
 * 16-byte aligned.  eqd_tn_partial_floats gives the size of `partial` (floats) and the chunking the kernel will use;
 * colsum needs nchunks * ncols floats.  Second stage: eqd_grad_reduce.                                               */
size_t eqd_tn_partial_floats(int64_t nrows, int32_t K, int32_t ncols, int32_t* rows_per_chunk_out, int32_t* nchunks_out);
int eqd_tn_gemm(const float* X, int32_t ldx, int32_t K, const float* D, int32_t ldd, int32_t ncols, int64_t nrows,
                float alpha, float* partial, float* colsum, int32_t* nchunks_out, void* stream);
/* grad[dst_index[i]] += sum_{c < nchunks} partial[c * stride + src_index[i]]   (fixed order, fp64 accumulation): the
 * deterministic second stage, and the scatter from the kernels' packed k-major panels to the state_dict layout.      */
int eqd_grad_reduce(const float* partial, int32_t nchunks, int64_t stride, const int32_t* src_index,
                    const int32_t* dst_index, int32_t n, float* grad, void* stream);

/* Node update backward (:319-337).  w_node1_lin = node_mlp.0.weight as [dhp][2 dhp + 136] (rows = hidden unit, columns
 * = the padded input blocks h | aggr | mu | h0(72)), w_node2_lin = node_mlp.4.weight as [64][dhp].  mu has row stride
 * ldmu.  Outputs: dh_in [n][dhp] (overwritten: skip path + h block), daggr [n][64], dmu [n][dhp], dh0_acc [n][72]
 * (accumulated), n5_out / du_out [n][dhp] (operands of the weight-gradient reductions), vec_partial
 * [n_partials][144] = per-CTA partials of {d node_mlp.3.weight [72], d node_mlp.3.bias [72]}.                          */
int eqd_bwd_node_mlp(const eqd_graph* g, const eqd_layer* p, const float* w_node1_lin, const float* w_node2_lin,
                     const float* h_in, int32_t ldh, const float* aggr, const float* mu, int32_t ldmu, const float* h0,
                     const float* dh_out, float* dh_in, float* daggr, float* dmu, float* dh0_acc, float* n5_out,
                     float* du_out, float* vec_partial /* [148][144] */, int32_t* n_partials_out, void* stream);
/* Same, regenerating the forward's site-2 mask of layer `layer` (dropout NULL = eqd_bwd_node_mlp). */
int eqd_bwd_node_mlp_dropout(const eqd_graph* g, const eqd_layer* p, const float* w_node1_lin, const float* w_node2_lin,
                             const float* h_in, int32_t ldh, const float* aggr, const float* mu, int32_t ldmu,
                             const float* h0, const float* dh_out, float* dh_in, float* daggr, float* dmu, float* dh0_acc,
                             float* n5_out, float* du_out, float* vec_partial, int32_t* n_partials_out,
                             const eqd_dropout* dropout, int32_t layer, void* stream);
/* Cross attention backward (:46-64, 247-256): dmu [n][dhp] -> dP[:, 128:] = [dQpre | dKpre | dV] of the combined
 * projection-gradient matrix dP [n][128 + 3 dhp].  proj = this layer's fp32 projections (eqd_project), mu the stashed
 * attention output, rowstat [n][4] scratch.                                                                         */
int eqd_bwd_attention(const eqd_graph* g, const eqd_layer* p, const float* proj, const float* mu, int32_t ldmu,
                      const float* dmu, float* dP, float* rowstat, void* stream);
/* Edge stage backward (:204-237, 263-292).  w2lin / w3lin = edge_mlp.4.weight / coors_mlp.0.weight [64][64] as in the
 * state_dict.  Outputs per edge: ein [E][44] = [he | rbf | 0 0], n1, msg, dz3, dmsg, dz1 [E][64], dxrel [E][3] (fp64);
 * vec_partial [n_partials][256] = per-CTA partials {d edge_mlp.3.weight [64], d edge_mlp.3.bias [64],
 * d coors_mlp.4.weight [64], d coors_mlp.4.bias [1]}.                                                                */
int eqd_bwd_edge(const eqd_graph* g, const eqd_layer* p, const float* w2lin, const float* w3lin, const float* proj,
                 const double* x_in, const float* daggr, const double* dx_out, float* ein_out, float* n1_out,
                 float* msg_out, float* dz3_out, float* dmsg_out, float* dz1_out, double* dxrel_out,
                 float* vec_partial /* [148][256] */, int32_t* n_partials_out, void* stream);
/* Same, regenerating the forward's site-0 / site-1 masks of layer `layer` (dropout NULL = eqd_bwd_edge). */
int eqd_bwd_edge_dropout(const eqd_graph* g, const eqd_layer* p, const float* w2lin, const float* w3lin, const float* proj,
                         const double* x_in, const float* daggr, const double* dx_out, float* ein_out, float* n1_out,
                         float* msg_out, float* dz3_out, float* dmsg_out, float* dz1_out, double* dxrel_out,
                         float* vec_partial, int32_t* n_partials_out, const eqd_dropout* dropout, int32_t layer,
                         void* stream);
/* Per node: dP[:, 0:64] = sum over OUT-edges of dz1, dP[:, 64:128] = sum over IN-edges, dx_in = (1 - eta) dx_out +
 * sum_out dxrel - sum_in dxrel.  out_ptr [n+1] / out_edge [E]: edges grouped by SOURCE node (ascending edge id).      */
int eqd_bwd_edge_gather(const eqd_graph* g, const int32_t* out_ptr, const int32_t* out_edge, const float* dz1,
                        const double* dxrel, const double* dx_out, float eta, float* dP, int32_t ldp, double* dx_in,
                        void* stream);
/* dh[n][0:dhp] += dP[n][:] . Wproj^T;  w_projT = eqd_layer_params.w_proj transposed, [128 + 3 dhp][dhp].            */
int eqd_bwd_project(const eqd_graph* g, const eqd_layer* p, const float* w_projT, const float* dP, float* dh,
                    void* stream);
/* d residue_emb_layer.weight [21][64] += sum over nodes of that residue type of (dh0_acc + dh_layer0)[0:64].         */
int eqd_bwd_embed(const eqd_graph* g, const float* res_lig, const float* res_rec, const float* dh0_acc,
                  const float* dh_layer0, float* demb, void* stream);
/* Keypoint read-out + Kabsch backward (:521-589, 657-665), fp64, incl. the 3x3 SVD backward (torch's svd_backward with
 * the guard's gap as denominator).  See csrc/head.cu for the argument semantics.                                      */
size_t eqd_bwd_head_workspace_bytes(int32_t n_nodes, int32_t n_node_tiles, int32_t n_pairs);
int eqd_bwd_head(const eqd_graph* g, const eqd_head_params* hp, const float* h, const double* x, const double* cov,
                 const float* x_lig_in, const float* dcoors, const double* dkeypts, const float* drot,
                 const float* dtrans, void* workspace, size_t workspace_bytes, float* dh, double* dx, float* dpre,
                 float* g_wkey, float* g_wquery, void* stream);
/* Same, regenerating the forward's site-3 mask; `layer` = the model's number of IEGMN layers (dropout NULL = eqd_bwd_head). */
int eqd_bwd_head_dropout(const eqd_graph* g, const eqd_head_params* hp, const float* h, const double* x, const double* cov,
                         const float* x_lig_in, const float* dcoors, const double* dkeypts, const float* drot,
                         const float* dtrans, void* workspace, size_t workspace_bytes, float* dh, double* dx, float* dpre,
                         float* g_wkey, float* g_wquery, const eqd_dropout* dropout, int32_t layer, void* stream);

/* ---- training losses on the device (src/train.py:41-49, 112-150; src/utils/ot_utils.py:5-29) ------------------------
 * Per pair: MSE of the predicted ligand coordinates, body-intersection loss, pocket OT loss with the EXACT earth mover's
 * distance (uniform marginals; successive shortest paths with potentials instead of POT's CPU network simplex), batch
 * means combined with the reference's weights; plus the gradients w.r.t. the predicted coordinates and the keypoints. */
size_t eqd_losses_workspace_bytes(int32_t n_rec_nodes, int32_t n_pocket_total);
int eqd_losses(const eqd_graph* g, const float* pred_lig /*[N_l][3]*/, const float* bound_lig /*[N_l][3]*/,
               const float* bound_rec /*[N_r][3]*/, const double* keypts /*[2B][50][3]*/,
               const int32_t* pocket_ptr /*[B+1]*/, const float* pocket_lig, const float* pocket_rec /*[sum P][3]*/,
               int32_t n_pocket_total, int32_t max_pocket /* largest pocket of the batch (host value; <= 1024) */,
               float pocket_ot_loss_weight, float intersection_loss_weight,
               float intersection_sigma, float intersection_surface_ct, void* workspace, size_t workspace_bytes,
               double* parts /*[B][4] mse, ot, intersection, -*/, double* total /*[4] loss, mse, ot, intersection*/,
               float* dcoors /*[N_l][3]*/, double* dkeypts /*[2B][50][3]*/, int32_t* err_flags, void* stream);

/* ---- residue k-NN graph construction on the device (src/utils/protein_utils.py:212-397, RBFs :71-86) ------------------
 * Proteins of a batch in engine order (ligand proteins of all pairs, then receptor proteins): seg_ptr [n_prot+1] residue
 * offsets, atom_ptr [n+1] atom offsets per residue, atoms [A][3] fp32 (all atoms, residue by residue), nca_c [n][3][3]
 * fp32 (N, CA, C of every residue), bound_ca [n][3] (bound-structure C-alpha trace the unbound one is aligned to; = CA
 * at inference).  Stage 1 writes deg [n], x [n][3] (ndata['x']), mu_r_norm [n][5]; the caller forms row_ptr = exclusive
 * prefix sum of deg (an index op) and calls stage 2, which writes col_src / edge_dst [E] (global node ids, grouped by
 * destination) and he [E][27].  `workspace` (eqd_graph_build_workspace_bytes) carries the fp64 aligned coordinates, local
 * frames and neighbour lists from stage 1 to stage 2.  max_neighbor <= 16.                                           */
size_t eqd_graph_build_workspace_bytes(int32_t n_nodes);
int eqd_graph_build_knn(int32_t n_prot, int32_t n_nodes, int32_t max_protein_nodes, const int32_t* seg_ptr,
                        const int32_t* atom_ptr, const float* atoms, const float* nca_c, const float* bound_ca, float cutoff,
                        int32_t max_neighbor, void* workspace, size_t workspace_bytes, int32_t* deg, float* x,
                        float* mu_r_norm, void* stream);
int eqd_graph_build_edges(int32_t n_nodes, const int32_t* row_ptr, const int32_t* deg, const void* workspace,
                          int32_t* col_src, int32_t* edge_dst, float* he, void* stream);

/* ---- batched RMSD meter (Meter_Unbound_Bound.update_rmsd, src/utils/eval.py:19-42; Kabsch src/utils/protein_utils.py:31-64) ----
 * out[b] = {complex RMSD after superimposing the predicted complex on the true one, ligand RMSD, receptor RMSD}, fp64.
 * Coordinates fp32, ligand arrays [N_l][3], receptor arrays [N_r][3] (receptor-local node order), batch order.        */
int eqd_rmsd_meter(const eqd_graph* g, const float* lig_pred, const float* rec_pred, const float* lig_true,
                   const float* rec_true, double* out /*[B][3]*/, void* stream);

/* ---- optimiser side on the flat fp32 parameter / gradient buffers (src/train.py:156, 165, 302) -----------------------
 * eqd_sqnorm_partials: partial[i] = sum of squares of slice i (n_partial <= 1024 doubles).  eqd_clip_adam: g *= scale_extra;
 * clip_grad_norm_(max_norm) with the global norm sqrt(sum partial) * |scale_extra|; torch.optim.Adam step (L2 weight decay,
 * bias correction at `step` >= 1); norm_out (device float, may be NULL) receives the pre-clip norm.                     */
int eqd_sqnorm_partials(const float* g, int64_t n, double* partial, int32_t n_partial, void* stream);
int eqd_clip_adam(float* w, float* g, float* m, float* v, int64_t n, const double* sq_partial, int32_t n_partial,
                  float max_norm, float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step,
                  float scale_extra, float* norm_out, void* stream);

void* eqd_event_create(void);
void eqd_event_destroy(void* event);
float eqd_event_elapsed_ms(void* begin, void* end);

#ifdef __cplusplus
}
#endif
#endif /* EQD_IEGMN_H */
