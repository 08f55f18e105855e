"""Drop-in replacement for the reference's ``src/model/rigid_docking_model.py`` whose arithmetic
runs in hand-written sm_100a CUDA kernels (``csrc/``) behind the C ABI of ``include/eqd_iegmn.h``.

Same public surface as the reference module (it is star-imported by ``src/utils/train_utils.py:14``,
which ``train.py`` / ``inference_rigid.py`` star-import in turn, so the module-level names ``nn``,
``math``, ``torch``, ``dgl``, ``fn``, ``sys`` are part of the contract):

* ``IEGMN_Layer(orig_h_feats_dim, h_feats_dim, out_feats_dim, fine_tune, args, log=None)``  (:83-91)
* ``IEGMN(args, n_lays, fine_tune, log=None)``                                              (:362)
* ``Rigid_Body_Docking_Net(args, log=None)`` / ``model(batch_hetero_graph, epoch)``          (:613, :642)
* ``compute_cross_attention``, ``get_mask``, ``get_non_lin``, ``get_layer_norm``,
  ``get_final_h_layer_norm``, ``apply_final_h_layer_norm``                                  (:10-78)

Parameter names and shapes equal the reference's ``state_dict`` (SURVEY 8b), so both shipped
checkpoints load with ``strict=True``.  The graph argument may be a batched DGL heterograph
(``train_utils.py:61-100``) or this package's DGL-free ``PairGraphBatch``.

Scope of this engine: forward AND backward of the configuration the shipped checkpoints use
(``nonlin='lkyrelu'``, ``layer_norm='LN'``, ``layer_norm_coors='0'``, ``final_h_layer_norm='0'``,
``cross_msgs``, ``use_dist_in_layers``, ``rot_model='kb_att'``, ``fine_tune=False``), with any ``dropout`` in [0, 1).
Anything else raises ``NotImplementedError``; a missing CUDA library raises -- there is no CPU path.
In training mode (``model.train()`` with grad enabled) the outputs of ``Rigid_Body_Docking_Net.forward`` are
autograd-connected: the whole path is one autograd node backed by the CUDA backward kernels (``training.py``).

Dropout: in ``train()`` mode with 0 < p < 1, ``Rigid_Body_Docking_Net.forward`` and ``IEGMN.forward`` apply the four
``nn.Dropout`` sites (edge_mlp, coors_mlp, node_mlp, mlp_h_mean_ROT), with or without grad enabled; p is read from the
``nn.Dropout`` modules at call time (they must agree).  Masks are counter-based (Philox4x32-10, ``include/eqd_iegmn.h``
``eqd_dropout``) under a 64-bit key drawn per call from torch's CUDA generator, so ``torch.manual_seed`` reproduces a run
and the CPU generator is left alone; they are statistically, not bitwise, torch's.  The per-layer operator
``IEGMN_Layer.forward`` and the inference tools (``graphed()``, ``serving``, ``graph_build``) keep raising
``NotImplementedError`` in that mode.
"""
import math  # noqa: F401  (re-exported, see module docstring)
import sys  # noqa: F401

import torch
from torch import nn

try:  # the real DGL when the reference's environment provides it
    import dgl
    from dgl import function as fn
except ImportError:  # DGL-free deployments use the package's own container
    from . import hetero_graph as dgl
    fn = None

from . import _native as nat
from .engine import GraphPlan, IEGMNEngine, PackedHead, PackedLayer, UnsortedEdges, _sorted_copy
from .hetero_graph import LIGAND, LL, RECEPTOR, RR


# ---- factory helpers (reference :10-42) --------------------------------------------------------

def get_non_lin(type, negative_slope):
    if type == 'swish':
        return nn.SiLU()
    assert type == 'lkyrelu'
    return nn.LeakyReLU(negative_slope=negative_slope)


def get_layer_norm(layer_norm_type, dim):
    if layer_norm_type == 'BN':
        return nn.BatchNorm1d(dim)
    if layer_norm_type == 'LN':
        return nn.LayerNorm(dim)
    return nn.Identity()


def get_final_h_layer_norm(layer_norm_type, dim):
    if layer_norm_type == 'BN':
        return nn.BatchNorm1d(dim)
    if layer_norm_type == 'LN':
        return nn.LayerNorm(dim)
    if layer_norm_type == 'GN':
        raise NotImplementedError("final_h_layer_norm='GN' is outside the CUDA engine's scope")
    assert layer_norm_type == '0'
    return nn.Identity()


def apply_final_h_layer_norm(g, h, node_type, norm_type, norm_layer):
    if norm_type == 'GN':
        return norm_layer(g, h, node_type)
    return norm_layer(h)


def get_mask(ligand_batch_num_nodes, receptor_batch_num_nodes, device):
    """Block-diagonal 0/1 mask of the reference's dense batched attention (:68-78).  Kept for API
    parity only: the engine's attention is segmented per pair and never materialises it."""
    rows, cols = int(sum(ligand_batch_num_nodes)), int(sum(receptor_batch_num_nodes))
    mask = torch.zeros(rows, cols, device=device)
    r = c = 0
    for l_n, r_n in zip(ligand_batch_num_nodes, receptor_batch_num_nodes):
        l_n, r_n = int(l_n), int(r_n)
        mask[r:r + l_n, c:c + r_n] = 1
        r, c = r + l_n, c + r_n
    return mask


def compute_cross_attention(queries, keys, values, mask, cross_msgs):
    """Dense masked attention with the reference's formula (:46-64), in plain torch ops.  API parity
    helper for callers outside the hot path; the engine itself uses the fused segmented kernel."""
    if not cross_msgs:
        return queries * 0.
    a = mask * torch.mm(queries, keys.t()) - 1000. * (1. - mask)
    return torch.mm(torch.softmax(a, dim=1), values)


# ---- shared host-side plumbing -------------------------------------------------------------------

_SUPPORTED = {'nonlin': 'lkyrelu', 'layer_norm': 'LN', 'layer_norm_coors': '0', 'final_h_layer_norm': '0',
              'cross_msgs': True, 'use_dist_in_layers': True}


def _check_layer_args(args):
    for k, v in _SUPPORTED.items():
        if args[k] != v:
            raise NotImplementedError(f"args[{k!r}]={args[k]!r}: the CUDA engine implements {v!r} only "
                                      '(the configuration of both shipped checkpoints)')


def _plan_for(graph, device, max_in_degree):
    """GraphPlan of a graph object, cached on it (the topology of a batch never changes)."""
    cached = getattr(graph, '_eqd_plan', None)
    if cached is not None and cached.device == device and cached.struct.max_in_degree == max_in_degree:
        return cached
    plan = GraphPlan.from_graph(graph, device, max_in_degree)
    try:
        graph._eqd_plan = plan
    except AttributeError:
        pass
    return plan


def _sorted_plan(graph, device, max_in_degree):
    src_l, dst_l = graph.edges(etype=LL)
    src_r, dst_r = graph.edges(etype=RR)
    args = (graph.batch_num_nodes(LIGAND).tolist(), graph.batch_num_nodes(RECEPTOR).tolist(), src_l.to(device),
            dst_l.to(device), src_r.to(device), dst_r.to(device), graph.edges[LL].data['he'].to(device),
            graph.edges[RR].data['he'].to(device), device, max_in_degree)
    plan = GraphPlan(*_sorted_copy(args))
    try:
        graph._eqd_plan = plan
    except AttributeError:
        pass
    return plan


def _module_state(module):
    return {k: v for k, v in module.state_dict(keep_vars=True).items()}


def _version_key(module):
    return tuple((p.data_ptr(), p._version) for p in module.parameters())


class IEGMN_Layer(nn.Module):
    """Parameters of one IEGMN layer (same names/shapes as the reference, :119-159) and its
    per-layer operator ``forward`` (:189-352) on the CUDA engine."""

    def __init__(self, orig_h_feats_dim, h_feats_dim, out_feats_dim, fine_tune, args, log=None):
        super().__init__()
        _check_layer_args(args)
        if fine_tune:
            raise NotImplementedError("fine_tune=True ('didn't work', args.py:110) is outside the engine's scope")
        edge_in = args['input_edge_feats_dim']
        drop, slope = args['dropout'], args['leakyrelu_neg_slope']
        act = lambda: get_non_lin(args['nonlin'], slope)
        self.cross_msgs = args['cross_msgs']
        self.final_h_layer_norm = args['final_h_layer_norm']
        self.use_dist_in_layers = args['use_dist_in_layers']
        self.skip_weight_h = args['skip_weight_h']
        self.x_connection_init = args['x_connection_init']
        self.leakyrelu_neg_slope = slope
        self.dropout_p = drop
        self.fine_tune = fine_tune
        self.debug, self.device, self.log = args['debug'], args['device'], log
        self.h_feats_dim, self.out_feats_dim = h_feats_dim, out_feats_dim
        self.graph_max_neighbor = int(args.get('graph_max_neighbor', 10) or 10)
        self.all_sigmas_dist = [1.5 ** x for x in range(15)]
        n_rbf = len(self.all_sigmas_dist)

        self.edge_mlp = nn.Sequential(nn.Linear(2 * h_feats_dim + edge_in + n_rbf, out_feats_dim), nn.Dropout(drop),
                                      act(), get_layer_norm(args['layer_norm'], out_feats_dim),
                                      nn.Linear(out_feats_dim, out_feats_dim))
        self.node_norm = nn.Identity()
        self.att_mlp_Q = nn.Sequential(nn.Linear(h_feats_dim, h_feats_dim, bias=False), act())
        self.att_mlp_K = nn.Sequential(nn.Linear(h_feats_dim, h_feats_dim, bias=False), act())
        self.att_mlp_V = nn.Sequential(nn.Linear(h_feats_dim, h_feats_dim, bias=False))
        self.node_mlp = nn.Sequential(nn.Linear(orig_h_feats_dim + 2 * h_feats_dim + out_feats_dim, h_feats_dim),
                                      nn.Dropout(drop), act(), get_layer_norm(args['layer_norm'], h_feats_dim),
                                      nn.Linear(h_feats_dim, out_feats_dim))
        self.final_h_layernorm_layer = get_final_h_layer_norm(self.final_h_layer_norm, out_feats_dim)
        self.coors_mlp = nn.Sequential(nn.Linear(out_feats_dim, out_feats_dim), nn.Dropout(drop), act(),
                                       get_layer_norm(args['layer_norm_coors'], out_feats_dim),
                                       nn.Linear(out_feats_dim, 1))
        if edge_in != nat.EDGE_FEATS or out_feats_dim != nat.HID or orig_h_feats_dim != nat.H0:
            raise NotImplementedError('CUDA engine widths: input_edge_feats_dim=27, hidden 64, node input 69')
        self._packed, self._packed_key = None, None

    def reset_parameters(self):
        for p in self.parameters():
            if p.dim() > 1:
                torch.nn.init.xavier_normal_(p, gain=1.)
            else:
                torch.nn.init.zeros_(p)

    def packed(self, device) -> PackedLayer:
        """Kernel-layout copy of the parameters, rebuilt only when a parameter changed."""
        key = (_version_key(self), str(device))
        if self._packed is None or self._packed_key != key:
            self._packed = PackedLayer(_module_state(self), device, float(self.skip_weight_h),
                                       float(self.x_connection_init), float(self.leakyrelu_neg_slope))
            self._packed_key = key
        return self._packed

    def _check_mode(self):
        if self.training and self.dropout_p > 0:
            raise NotImplementedError('dropout > 0 in training mode is not implemented in the CUDA engine')

    def forward(self, hetero_graph, coors_ligand, h_feats_ligand, original_ligand_node_features,
                original_edge_feats_ligand, orig_coors_ligand, coors_receptor, h_feats_receptor,
                original_receptor_node_features, original_edge_feats_receptor, orig_coors_receptor):
        """Per-layer operator with the reference's signature and return value
        ``(x_final_ligand, node_upd_ligand, x_final_receptor, node_upd_receptor)``."""
        import ctypes as C
        self._check_mode()
        dev = coors_ligand.device
        eng = IEGMNEngine(dev)
        plan = _plan_for(hetero_graph, dev, self.graph_max_neighbor)
        if original_edge_feats_ligand.data_ptr() != plan.he_l.data_ptr():  # caller scaled / replaced he
            plan = GraphPlan(plan.n_lig_list, plan.n_rec_list, *hetero_graph.edges(etype=LL),
                             *hetero_graph.edges(etype=RR), original_edge_feats_ligand, original_edge_feats_receptor,
                             dev, self.graph_max_neighbor)
        lay = self.packed(dev)
        N, dhp = plan.N, lay.dhp
        f32, f64 = dict(dtype=torch.float32, device=dev), dict(dtype=torch.float64, device=dev)
        h = torch.zeros(N, dhp, **f32)
        h[:, :lay.dh] = torch.cat([h_feats_ligand, h_feats_receptor]).to(**f32)
        h0 = torch.zeros(N, nat.H0_PAD, **f32)
        h0[:, :nat.H0] = torch.cat([original_ligand_node_features, original_receptor_node_features]).to(**f32)
        x_in = torch.cat([coors_ligand, coors_receptor]).to(**f64).contiguous()
        x_orig = torch.cat([orig_coors_ligand, orig_coors_receptor]).to(**f64).contiguous()
        proj = torch.empty(N, 128 + 3 * dhp, **f32)
        aggr, h_out = torch.empty(N, nat.HID, **f32), torch.empty(N, nat.HID, **f32)
        x_out = torch.empty(N, 3, **f64)
        status = torch.zeros(plan.n_pairs + 1, dtype=torch.int32, device=dev)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        g, lp = C.byref(plan.struct), C.byref(lay.struct)
        nat.check(eng.lib.eqd_project(g, lp, nat.ptr(h), dhp, nat.ptr(proj), st), 'eqd_project')
        nat.check(eng.lib.eqd_iegmn_layer_forward(g, lp, None, nat.ptr(h), dhp, nat.ptr(h0), nat.ptr(x_in),
                                                  nat.ptr(x_orig), nat.ptr(proj), None, nat.ptr(aggr), nat.ptr(h_out),
                                                  nat.ptr(x_out), nat.ptr(status), st), 'eqd_iegmn_layer_forward')
        if int(status[plan.n_pairs].item()) & nat.STATUS_DEGREE_OVERFLOW or bool(plan.unsorted.item()):
            raise nat.NativeLibraryError('IEGMN_Layer.forward: edges must be grouped by destination with in-degree '
                                         f'<= {self.graph_max_neighbor}')
        x_out = x_out.to(coors_ligand.dtype)
        return x_out[:plan.N_l], h_out[:plan.N_l], x_out[plan.N_l:], h_out[plan.N_l:]

    def __repr__(self):
        return 'IEGMN Layer (B200 engine) ' + str({k: v for k, v in self.__dict__.items() if not k.startswith('_')})


class IEGMN(nn.Module):
    """Embedding + IEGMN layer stack + keypoint attention + Kabsch (reference :360-606)."""

    def __init__(self, args, n_lays, fine_tune, log=None):
        super().__init__()
        self.debug, self.log = args['debug'], log
        self.device = args['device']
        self.graph_nodes = args['graph_nodes']
        self.rot_model = args['rot_model']
        self.noise_decay_rate, self.noise_initial = args['noise_decay_rate'], args['noise_initial']
        self.use_edge_features_in_gmn = args['use_edge_features_in_gmn']
        self.use_mean_node_features = args['use_mean_node_features']
        self.leakyrelu_neg_slope = args['leakyrelu_neg_slope']
        self.graph_max_neighbor = int(args.get('graph_max_neighbor', 10) or 10)
        assert self.graph_nodes == 'residues'
        assert args['rot_model'] == 'kb_att'
        if not (self.use_edge_features_in_gmn and self.use_mean_node_features):
            raise NotImplementedError('CUDA engine: use_edge_features_in_gmn and use_mean_node_features must be on')

        if int(args['residue_emb_dim']) != nat.HID:
            raise NotImplementedError(f'CUDA engine: residue_emb_dim must be {nat.HID}')
        self.residue_emb_layer = nn.Embedding(num_embeddings=21, embedding_dim=args['residue_emb_dim'])
        in_dim = args['residue_emb_dim'] + 5  # + mu_r_norm surface features (:387-388)
        hid = args['iegmn_lay_hid_dim']
        self.iegmn_layers = nn.ModuleList()
        self.iegmn_layers.append(IEGMN_Layer(in_dim, in_dim, hid, fine_tune, args, log))
        if args['shared_layers']:
            shared = IEGMN_Layer(in_dim, hid, hid, fine_tune, args, log)
            for _ in range(1, n_lays):
                self.iegmn_layers.append(shared)
        else:
            for _ in range(1, n_lays):
                self.iegmn_layers.append(IEGMN_Layer(in_dim, hid, hid, fine_tune, args, log))

        self.num_att_heads = args['num_att_heads']
        self.out_feats_dim = hid
        if self.num_att_heads != nat.HEADS:
            raise NotImplementedError(f'CUDA engine: num_att_heads must be {nat.HEADS}')
        self.att_mlp_key_ROT = nn.Sequential(nn.Linear(hid, self.num_att_heads * hid, bias=False))
        self.att_mlp_query_ROT = nn.Sequential(nn.Linear(hid, self.num_att_heads * hid, bias=False))
        self.mlp_h_mean_ROT = nn.Sequential(nn.Linear(hid, hid), nn.Dropout(args['dropout']),
                                            get_non_lin(args['nonlin'], args['leakyrelu_neg_slope']))
        self._head, self._head_key = None, None
        self.last_outputs = None

    def reset_parameters(self):
        for p in self.parameters():
            if p.dim() > 1:
                torch.nn.init.xavier_normal_(p, gain=1.)
            else:
                torch.nn.init.zeros_(p)

    def packed_head(self, device) -> PackedHead:
        mods = (self.att_mlp_key_ROT, self.att_mlp_query_ROT, self.mlp_h_mean_ROT)
        key = (tuple(_version_key(m) for m in mods), str(device))
        if self._head is None or self._head_key != key:
            self._head = PackedHead(self.mlp_h_mean_ROT[0].weight, self.mlp_h_mean_ROT[0].bias,
                                    self.att_mlp_key_ROT[0].weight, self.att_mlp_query_ROT[0].weight, device,
                                    float(self.leakyrelu_neg_slope))
            self._head_key = key
        return self._head

    def dropout_p(self) -> float:
        """The dropout probability the next forward applies: p of the model's ``nn.Dropout`` modules that are in training
        mode (0 when none is).  Raises NotImplementedError when active modules disagree or p >= 1."""
        mods = [m for lay in self.iegmn_layers for m in (lay.edge_mlp[1], lay.coors_mlp[1], lay.node_mlp[1])]
        mods.append(self.mlp_h_mean_ROT[1])
        ps = {float(m.p) if m.training else 0.0 for m in mods}
        if len(ps) > 1:
            raise NotImplementedError(f'dropout probabilities / modes differ between the nn.Dropout modules ({sorted(ps)}): '
                                      'the CUDA engine applies one p to all four sites')
        p = ps.pop()
        if p >= 1.0:
            raise NotImplementedError(f'dropout p={p} >= 1 is not implemented in the CUDA engine')
        return p

    def run_engine(self, batch_hetero_graph, check_status=True, record_event=True, allow_dropout=False):
        """The whole hot path on the device; returns the engine's raw output dict.  With ``check_status=False`` the
        per-pair status words are left pending (``resolve(out)`` finishes the call).  ``record_event=False`` is for
        CUDA-graph capture (``graphed.GraphedForward``), which records its own completion event per replay.
        ``allow_dropout`` (``IEGMN.forward``): apply dropout in train() mode; otherwise that mode raises, as in the
        inference tools built on this call."""
        emb = self.residue_emb_layer.weight
        dev = emb.device
        drop_p = 0.0
        if allow_dropout:
            drop_p = self.dropout_p()
        else:
            for lay in self.iegmn_layers:
                lay._check_mode()
        eng = IEGMNEngine(dev)
        layers = [lay.packed(dev) for lay in self.iegmn_layers]
        head = self.packed_head(dev)
        nl, nr = batch_hetero_graph.nodes[LIGAND].data, batch_hetero_graph.nodes[RECEPTOR].data
        plan = _plan_for(batch_hetero_graph, dev, self.graph_max_neighbor)
        emb32 = emb.detach().to(torch.float32).contiguous()
        call = lambda p, chk: eng.forward(p, emb32, layers, head, nl['res_feat'], nr['res_feat'], nl['mu_r_norm'],
                                          nr['mu_r_norm'], nl['new_x'], nr['x'], chk, self.log,
                                          record_event=record_event, dropout_p=drop_p)
        try:
            out = call(plan, check_status)
        except UnsortedEdges:
            plan = _sorted_plan(batch_hetero_graph, dev, self.graph_max_neighbor)
            out = call(plan, True)
        out['plan'], out['engine'], out['graph'] = plan, eng, batch_hetero_graph
        out['allow_dropout'] = allow_dropout
        return out

    def resolve(self, out):
        """Finishes a ``run_engine(..., check_status=False)`` call: waits for its status words and replays the
        reference's host-side control flow for flagged pairs (:570-584).  Unsorted edge lists are re-run sorted."""
        try:
            out['engine'].resolve_status(out['plan'], out, out['kabsch'], self.log)
            return out
        except UnsortedEdges:
            return self.run_engine(out['graph'], True, allow_dropout=out.get('allow_dropout', False))

    def forward(self, batch_hetero_graph, epoch):
        """Returns ``[T list, b list, Y_ligand list, Y_receptor list]`` like the reference (:602) and
        writes ``x_iegmn_out`` / ``hv_iegmn_out`` into the graph (:507-510).  Applies dropout in train() mode."""
        return self.package(self.run_engine(batch_hetero_graph, allow_dropout=True), batch_hetero_graph)

    def package(self, out, batch_hetero_graph):
        plan = out['plan']
        B, N_l = plan.n_pairs, plan.N_l
        dt = batch_hetero_graph.nodes[LIGAND].data['new_x'].dtype
        x_fin = out['x64'].to(dt)
        nl, nr = batch_hetero_graph.nodes[LIGAND].data, batch_hetero_graph.nodes[RECEPTOR].data
        nl['x_iegmn_out'], nr['x_iegmn_out'] = x_fin[:N_l], x_fin[N_l:]
        nl['hv_iegmn_out'], nr['hv_iegmn_out'] = out['h'][:N_l], out['h'][N_l:]
        keyp = out['keypts'].to(dt)
        self.last_outputs = out
        return [list(out['rotation'].unbind(0)), list(out['translation'].unbind(0)),
                list(keyp[:B].unbind(0)), list(keyp[B:].unbind(0))]

    def __repr__(self):
        return 'IEGMN (B200 engine) ' + str({k: v for k, v in self.__dict__.items() if not k.startswith('_')})


class Rigid_Body_Docking_Net(nn.Module):
    """``model(batch_hetero_graph, epoch)`` -> (ligand coords list, ligand keypoints list, receptor
    keypoints list, rotations list, translations list), reference :611-696."""

    def __init__(self, args, log=None):
        super().__init__()
        self.debug, self.log, self.device = args['debug'], log, args['device']
        if args['fine_tune']:
            raise NotImplementedError("fine_tune=True is outside the CUDA engine's scope (both checkpoints: fine_F)")
        self.iegmn_original = IEGMN(args, n_lays=args['iegmn_n_lays'], fine_tune=False, log=log)
        self.list_iegmns = [('finetune', self.iegmn_original)]

    def reset_parameters(self):
        for p in self.parameters():
            if p.dim() > 1:
                torch.nn.init.xavier_normal_(p, gain=1.)
            else:
                torch.nn.init.zeros_(p)

    def forward_async(self, batch_hetero_graph, epoch=0):
        """Launches the whole forward without waiting for its status words; ``.result()`` of the returned handle
        completes it and returns the reference's 5-tuple.  Lets a serving loop keep several batches in flight."""
        net, raw = self, self.iegmn_original.run_engine(batch_hetero_graph, check_status=False)

        class Pending:
            def raw_result(self_inner):
                """The engine's batched output dict (``ligand_coors`` (sum N_l, 3), ``rotation`` (B, 3, 3),
                ``translation`` (B, 1, 3), ``keypts`` (2B, 50, 3), ...) once the status words are resolved."""
                return net.iegmn_original.resolve(raw)

            def result(self_inner):
                out = net.iegmn_original.resolve(raw)
                return net._assemble(net.iegmn_original.package(out, batch_hetero_graph))
        return Pending()

    def graphed(self, device_batch):
        """A CUDA-graph capture of this model's forward for one fixed-shape device batch (``graphed.GraphedForward``):
        ``.launch().result()`` returns what ``model(batch, epoch)`` returns at the host cost of one graph launch."""
        from .graphed import GraphedForward
        return GraphedForward(self, device_batch)

    def forward(self, batch_hetero_graph, epoch):
        if (self.training or getattr(self, 'force_autograd', False)) and torch.is_grad_enabled():
            return self._forward_autograd(batch_hetero_graph)
        return self._assemble(self.iegmn_original(batch_hetero_graph, epoch))

    def _forward_autograd(self, batch_hetero_graph):
        """Training mode (``model.train()``, src/train.py:64): the whole hot path is ONE autograd node whose backward is the
        hand-written CUDA backward (``training.TrainEngine``), so ``loss.backward()`` (train.py:154) fills ``param.grad`` of
        every parameter exactly like the reference's autograd graph does.  Outputs are autograd-connected views of the
        node's four raw outputs.  Evaluation under ``torch.no_grad()`` / ``model.eval()`` keeps the inference path."""
        from .training import autograd_forward
        fwd, (coors, keypts, rot, trans) = autograd_forward(self, batch_hetero_graph, self.log)
        plan = fwd['plan']
        B, N_l = plan.n_pairs, plan.N_l
        nl, nr = batch_hetero_graph.nodes[LIGAND].data, batch_hetero_graph.nodes[RECEPTOR].data
        dt = nl['new_x'].dtype
        x_fin = fwd['x64'].to(dt)
        nl['x_iegmn_out'], nr['x_iegmn_out'] = x_fin[:N_l], x_fin[N_l:]
        nl['hv_iegmn_out'], nr['hv_iegmn_out'] = fwd['h'][:N_l], fwd['h'][N_l:]
        self.iegmn_original.last_outputs = fwd
        keyp = keypts.to(dt)
        return (list(torch.split(coors, plan.n_lig_list, dim=0)), list(keyp[:B].unbind(0)), list(keyp[B:].unbind(0)),
                list(rot.unbind(0)), list(trans.unbind(0)))

    def _assemble(self, outputs):
        assert len(outputs) == 4
        raw = self.iegmn_original.last_outputs
        plan = raw['plan']
        # T new_x + b of every ligand node was applied by the Kabsch kernel (:665)
        ligand_coors = list(torch.split(raw['ligand_coors'], plan.n_lig_list, dim=0))
        for b_align in outputs[1]:
            assert b_align.shape[0] == 1 and b_align.shape[1] == 3
        return ligand_coors, outputs[2], outputs[3], outputs[0], outputs[1]

    def __repr__(self):
        return 'Rigid_Body_Docking_Net (B200 engine) ' + str({k: v for k, v in self.__dict__.items()
                                                              if not k.startswith('_')})
