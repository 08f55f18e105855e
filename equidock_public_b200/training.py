"""Training side of the B200 engine: forward with a layer stash, the hand-written backward (csrc/bwd_*.cu, head.cu,
losses.cu) driven over the C ABI, a ``torch.autograd.Function`` so that the reference's own training loop
(``loss.backward()``, src/train.py:154) works on the drop-in module unchanged, and a fused data-parallel trainer
(device losses, flat-gradient NCCL all-reduce overlapped with the tail of backward, clip + Adam in one kernel;
src/train.py:98-165, 302).

PyTorch is plumbing here too: device memory, streams, ``torch.distributed``; a few index ops build the by-source edge
permutation once per batch topology.  No gradient arithmetic is done by torch.  There is no CPU fallback.

Gradient layout: ONE flat fp32 buffer holding every unique parameter in the order [head, layer L-1, ..., layer 0,
embedding] (the order the backward finishes them in, so that all-reduce buckets are contiguous and can start while
earlier layers are still being differentiated); ``param.grad`` tensors are views of it.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _native as nat
from .engine import GraphPlan, IEGMNEngine, PackedHead, PackedLayer, _StatusLease, _upload_blob, _host_f32

_f32 = torch.float32


class ParamLayout:
    """Flat layout of a model's unique parameters in backward-completion order."""

    def __init__(self, model):
        iegmn = model.iegmn_original
        seen, self.entries = set(), []          # (qualified name, param)
        self.buckets: List[tuple] = []          # (label, lo, hi) contiguous slices, in completion order
        self.module_bucket: Dict[int, str] = {}  # id(layer module) -> its bucket label
        self.total = 0
        self._offs: List[int] = []

        def add(prefix, module, label):
            lo = self.total
            for n, p in module.named_parameters():
                if id(p) in seen:
                    continue
                seen.add(id(p))
                self.entries.append((f'{prefix}{n}', p))
                self._offs.append(self.total)
                self.total += (p.numel() + 63) & ~63       # every parameter starts on a 256-byte boundary: the kernels
                                                           # read weights 16 bytes at a time straight from the flat buffer
            if self.total > lo:
                self.buckets.append((label, lo, self.total))
                self.module_bucket[id(module)] = label

        add('iegmn_original.att_mlp_key_ROT.', iegmn.att_mlp_key_ROT, 'head')
        add('iegmn_original.att_mlp_query_ROT.', iegmn.att_mlp_query_ROT, 'head')
        add('iegmn_original.mlp_h_mean_ROT.', iegmn.mlp_h_mean_ROT, 'head')
        # merge the three head modules into one bucket
        self.buckets = [('head', 0, self.total)]
        for li in reversed(range(len(iegmn.iegmn_layers))):
            add(f'iegmn_original.iegmn_layers.{li}.', iegmn.iegmn_layers[li], f'layer{li}')
        add('iegmn_original.residue_emb_layer.', iegmn.residue_emb_layer, 'emb')
        self.offset: Dict[int, int] = {}
        self.name_offset: Dict[str, int] = {}
        for (name, p), o in zip(self.entries, self._offs):
            self.offset[id(p)] = o
            self.name_offset[name] = o
        self.params = [p for _, p in self.entries]
        self.n_param_elements = sum(p.numel() for p in self.params)

    def views(self, flat: torch.Tensor) -> List[torch.Tensor]:
        return [flat[self.offset[id(p)]:self.offset[id(p)] + p.numel()].view(p.shape) for p in self.params]


def _i32(a, device):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(device)


class LayerTrainPack:
    """Backward-side tensors of one IEGMN_Layer module: the nn.Linear-layout weight panels the data-gradient GEMMs
    read, and the (source index, destination index) maps of every weight-gradient reduction (packed k-major partial ->
    flat state_dict-layout gradient)."""

    def __init__(self, layer_module, packed: PackedLayer, layout: ParamLayout, device, maps=None):
        dh, dhp = packed.dh, packed.dhp
        pw = 128 + 3 * dhp
        win = 2 * dhp + 64 + nat.H0_PAD
        sd = {k: _host_f32(v) for k, v in layer_module.state_dict(keep_vars=True).items()}
        w5, w6 = sd['node_mlp.0.weight'], sd['node_mlp.4.weight']
        w1lin = torch.zeros(dhp, win)
        w1lin[:dh, 0:dh] = w5[:, 0:dh]
        w1lin[:dh, dhp:dhp + 64] = w5[:, dh:dh + 64]
        w1lin[:dh, dhp + 64:dhp + 64 + dh] = w5[:, dh + 64:2 * dh + 64]
        w1lin[:dh, 2 * dhp + 64:2 * dhp + 64 + nat.H0] = w5[:, 2 * dh + 64:]
        w2lin = torch.zeros(64, dhp)
        w2lin[:, :dh] = w6
        self.t = _upload_blob({'w_node1_lin': w1lin, 'w_node2_lin': w2lin,
                               'w_projT': packed.t['w_proj'].detach().cpu().t().contiguous(),
                               'w2lin': sd['edge_mlp.4.weight'].contiguous(),
                               'w3lin': sd['coors_mlp.0.weight'].contiguous()}, device)
        self.dh, self.dhp, self.pw = dh, dhp, pw
        if maps is not None:           # the index maps depend on the layout only: built once per module
            self.maps = maps
            return
        off = {n: layout.offset[id(p)] for n, p in layer_module.named_parameters()}
        ein = 2 * dh + 42
        w1n = 2 * dh + 64 + nat.H0            # node_mlp.0 input width
        kk, nn = np.meshgrid(np.arange(dh), np.arange(64), indexing='ij')     # k = input feature, n = output unit

        def m(src, dst):
            return _i32(np.asarray(src).reshape(-1), device), _i32(np.asarray(dst).reshape(-1), device)

        maps = {}
        # (a) projections: partial [dhp][pw], colsum [pw]
        src, dst = [], []
        src.append(kk * pw + nn); dst.append(off['edge_mlp.0.weight'] + nn * ein + kk)                  # Psrc block
        src.append(kk * pw + 64 + nn); dst.append(off['edge_mlp.0.weight'] + nn * ein + dh + kk)        # Pdst block
        k2, c2 = np.meshgrid(np.arange(dh), np.arange(dh), indexing='ij')
        for gi, name in enumerate(('att_mlp_Q.0.weight', 'att_mlp_K.0.weight', 'att_mlp_V.0.weight')):
            src.append(k2 * pw + 128 + gi * dhp + c2); dst.append(off[name] + c2 * dh + k2)
        maps['proj'] = m(np.concatenate([a.reshape(-1) for a in src]), np.concatenate([a.reshape(-1) for a in dst]))
        maps['proj_bias'] = m(64 + np.arange(64), off['edge_mlp.0.bias'] + np.arange(64))
        # (b) edge GEMM1: partial [44][64]
        k42, n64 = np.meshgrid(np.arange(42), np.arange(64), indexing='ij')
        maps['edge1'] = m(k42 * 64 + n64, off['edge_mlp.0.weight'] + n64 * ein + 2 * dh + k42)
        k64, n64b = np.meshgrid(np.arange(64), np.arange(64), indexing='ij')
        maps['edge2'] = m(k64 * 64 + n64b, off['edge_mlp.4.weight'] + n64b * 64 + k64)
        maps['edge2_bias'] = m(np.arange(64), off['edge_mlp.4.bias'] + np.arange(64))
        maps['edge3'] = m(k64 * 64 + n64b, off['coors_mlp.0.weight'] + n64b * 64 + k64)
        maps['edge3_bias'] = m(np.arange(64), off['coors_mlp.0.bias'] + np.arange(64))
        maps['edgevec'] = m(np.concatenate([np.arange(64), 64 + np.arange(64), 128 + np.arange(64), [192]]),
                            np.concatenate([off['edge_mlp.3.weight'] + np.arange(64), off['edge_mlp.3.bias'] + np.arange(64),
                                            off['coors_mlp.4.weight'] + np.arange(64), [off['coors_mlp.4.bias']]]))
        # node MLP layer 1: four TN products against du [N][dhp] -> partial [K][dhp]
        kh, nh = np.meshgrid(np.arange(dh), np.arange(dh), indexing='ij')
        maps['node_h'] = m(kh * dhp + nh, off['node_mlp.0.weight'] + nh * w1n + kh)
        ka, na = np.meshgrid(np.arange(64), np.arange(dh), indexing='ij')
        maps['node_aggr'] = m(ka * dhp + na, off['node_mlp.0.weight'] + na * w1n + dh + ka)
        maps['node_mu'] = m(kh * dhp + nh, off['node_mlp.0.weight'] + nh * w1n + dh + 64 + kh)
        k0, n0 = np.meshgrid(np.arange(nat.H0), np.arange(dh), indexing='ij')
        maps['node_h0'] = m(k0 * dhp + n0, off['node_mlp.0.weight'] + n0 * w1n + 2 * dh + 64 + k0)
        maps['node1_bias'] = m(np.arange(dh), off['node_mlp.0.bias'] + np.arange(dh))
        kn, nn2 = np.meshgrid(np.arange(dh), np.arange(64), indexing='ij')
        maps['node2'] = m(kn * 64 + nn2, off['node_mlp.4.weight'] + nn2 * dh + kn)
        maps['node2_bias'] = m(np.arange(64), off['node_mlp.4.bias'] + np.arange(64))
        maps['nodevec'] = m(np.concatenate([np.arange(dh), 72 + np.arange(dh)]),
                            np.concatenate([off['node_mlp.3.weight'] + np.arange(dh), off['node_mlp.3.bias'] + np.arange(dh)]))
        self.maps = maps


class BackwardWorkspace:
    """Device buffers of one backward, sized for a plan (reused across steps with the same sizes)."""

    def __init__(self, plan: GraphPlan, device):
        N, E, B = plan.N, plan.E, plan.n_pairs
        f = lambda *s: torch.empty(*s, dtype=_f32, device=device)
        d = lambda *s: torch.empty(*s, dtype=torch.float64, device=device)
        self.key = (N, E, B)
        self.proj, self.dP = f(N, 344), f(N, 344)
        self.dh = [f(N, 72), f(N, 72)]
        self.dx = [d(N, 3), d(N, 3)]
        self.daggr, self.dmu, self.dh0 = f(N, 64), f(N, 72), f(N, 72)
        self.n5, self.du, self.rowstat, self.dpre = f(N, 72), f(N, 72), f(N, 4), f(N, 64)
        self.ein = f(max(E, 1), 44)
        self.n1, self.msg, self.dz3, self.dmsg, self.dz1 = (f(max(E, 1), 64) for _ in range(5))
        self.dxrel = d(max(E, 1), 3)
        lib = nat.load()
        need = 0
        for rows, K, nc in ((E, 64, 64), (E, 44, 64), (N, 72, 344), (N, 72, 72), (N, 72, 64)):
            need = max(need, int(lib.eqd_tn_partial_floats(rows, K, nc, None, None)))
        self.partial = f(max(need, 1))
        self.colsum = f(4096 * 344)
        self.vec = f(148 * 256)
        self.head_ws_bytes = int(lib.eqd_bwd_head_workspace_bytes(N, plan.n_node_tiles, B))
        self.head_ws = torch.empty(self.head_ws_bytes, dtype=torch.uint8, device=device)
        # edges grouped by SOURCE node (ascending edge id inside a group): the transpose index of the CSR-by-destination
        order = torch.sort(plan.col_src.long(), stable=True)
        self.out_edge = order.indices.to(torch.int32).contiguous()
        self.out_ptr = torch.searchsorted(order.values.to(torch.int32).contiguous(),
                                          torch.arange(N + 1, dtype=torch.int32, device=device), out_int32=True).contiguous()


class TrainEngine:
    """Forward-with-stash and backward of one model on one device."""

    def __init__(self, model):
        self.model = model
        self.iegmn = model.iegmn_original
        self.device = self.iegmn.residue_emb_layer.weight.device
        if self.device.type != 'cuda':
            raise nat.NativeLibraryError('training runs on a CUDA device only (no CPU fallback)')
        self.lib = nat.load()
        self.layout = ParamLayout(model)
        self._packs: Dict[int, tuple] = {}
        self._maps: Dict[int, dict] = {}
        self._ws: Optional[BackwardWorkspace] = None
        self._head_maps = None
        self.rank = 0   # data-parallel rank: the fourth word of the dropout counter (DataParallelTrainer sets it)

    # ---- packs ----------------------------------------------------------------------------------------------------
    def layer_pack(self, lay_module) -> LayerTrainPack:
        packed = lay_module.packed(self.device)
        hit = self._packs.get(id(lay_module))
        if hit is None or hit[0] is not packed:
            maps = self._maps.get(id(lay_module))
            tp = LayerTrainPack(lay_module, packed, self.layout, self.device, maps)
            self._maps[id(lay_module)] = tp.maps
            hit = (packed, tp)
            self._packs[id(lay_module)] = hit
        return hit[1]

    def head_maps(self):
        if self._head_maps is None:
            off = self.layout.name_offset
            k, n = np.meshgrid(np.arange(64), np.arange(64), indexing='ij')
            self._head_maps = {
                'wm': (_i32((k * 64 + n).reshape(-1), self.device),
                       _i32((off['iegmn_original.mlp_h_mean_ROT.0.weight'] + n * 64 + k).reshape(-1), self.device)),
                'bm': (_i32(np.arange(64), self.device),
                       _i32(off['iegmn_original.mlp_h_mean_ROT.0.bias'] + np.arange(64), self.device))}
        return self._head_maps

    # ---- forward with stash -----------------------------------------------------------------------------------------
    def forward(self, graph, log=None):
        from .rigid_docking_model import _plan_for, _sorted_plan, UnsortedEdges
        iegmn, dev, lib = self.iegmn, self.device, self.lib
        p = iegmn.dropout_p()   # > 0 in train() mode with dropout: masks drawn per call, regenerated by backward()
        plan = _plan_for(graph, dev, iegmn.graph_max_neighbor)
        try:
            return self._forward_plan(graph, plan, log, p)
        except UnsortedEdges:
            return self._forward_plan(graph, _sorted_plan(graph, dev, iegmn.graph_max_neighbor), log, p)

    def _forward_plan(self, graph, plan, log, dropout_p=0.0):
        from .hetero_graph import LIGAND, RECEPTOR
        iegmn, dev, lib = self.iegmn, self.device, self.lib
        layers = [lay.packed(dev) for lay in iegmn.iegmn_layers]
        head = iegmn.packed_head(dev)
        nl, nr = graph.nodes[LIGAND].data, graph.nodes[RECEPTOR].data
        L = len(layers)
        with torch.cuda.device(dev):
            g = C.byref(plan.struct)
            stash_bytes = int(lib.eqd_forward_stash_bytes(g, L))
            offs = (C.c_size_t * 9)()
            nat.check(lib.eqd_forward_stash_offsets(g, L, offs), 'eqd_forward_stash_offsets')
            stash = torch.empty(stash_bytes, dtype=torch.uint8, device=dev)
            eng = IEGMNEngine(dev)
            emb32 = iegmn.residue_emb_layer.weight.detach().to(_f32).contiguous()
            out = eng.forward(plan, emb32, layers, head, nl['res_feat'], nr['res_feat'], nl['mu_r_norm'], nr['mu_r_norm'],
                              nl['new_x'], nr['x'], True, log, train_stash=stash, dropout_p=dropout_p,
                              dropout_rank=self.rank)
        out.update(plan=plan, engine=eng, graph=graph, stash=stash, stash_offsets=list(offs), layers=layers, head=head,
                   res_l=nl['res_feat'].to(_f32).contiguous(), res_r=nr['res_feat'].to(_f32).contiguous(),
                   x_lig_in=nl['new_x'].to(_f32).contiguous())
        return out

    # ---- backward -------------------------------------------------------------------------------------------------
    def _tn(self, ws, X, ldx, K, D, ldd, ncols, nrows, alpha, want_colsum, st):
        nch = C.c_int32(0)
        nat.check(self.lib.eqd_tn_gemm(nat.ptr(X), ldx, K, nat.ptr(D), ldd, ncols, nrows, alpha, nat.ptr(ws.partial),
                                       nat.ptr(ws.colsum) if want_colsum else None, C.byref(nch), st), 'eqd_tn_gemm')
        return nch.value

    def _reduce(self, src_t, nch, stride, mp, flat, st):
        nat.check(self.lib.eqd_grad_reduce(nat.ptr(src_t), nch, stride, nat.ptr(mp[0]), nat.ptr(mp[1]), int(mp[0].numel()),
                                           nat.ptr(flat), st), 'eqd_grad_reduce')

    def backward(self, fwd, d_coors, d_keypts, d_rot=None, d_trans=None, flat: Optional[torch.Tensor] = None,
                 on_bucket_done=None, capture: Optional[list] = None) -> torch.Tensor:
        """Gradients of every parameter for upstream gradients w.r.t. the four raw outputs (ligand coordinates
        (N_l,3) f32, keypoints (2B,50,3) f64, rotations (B,3,3) f32, translations (B,1,3) f32; any may be None).
        Returns the flat gradient buffer (see ParamLayout).  ``on_bucket_done(label, lo, hi)`` is called on the host
        right after the kernels that complete a bucket have been queued (the data-parallel trainer launches that
        bucket's all-reduce there)."""
        lib, dev, lay_out = self.lib, self.device, self.layout
        plan: GraphPlan = fwd['plan']
        iegmn = self.iegmn
        N, E, B = plan.N, plan.E, plan.n_pairs
        L = len(fwd['layers'])
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            if self._ws is None or self._ws.key != (N, E, B) or self._ws_plan is not plan:
                self._ws = BackwardWorkspace(plan, dev)
                self._ws_plan = plan
            ws = self._ws
            if flat is None:
                flat = torch.zeros(lay_out.total, dtype=_f32, device=dev)
            g = C.byref(plan.struct)
            cf = lambda t, dt: None if t is None else t.detach().to(device=dev, dtype=dt).contiguous()
            d_coors, d_rot, d_trans = cf(d_coors, _f32), cf(d_rot, _f32), cf(d_trans, _f32)
            d_keypts = cf(d_keypts, torch.float64)
            off = lay_out.name_offset
            gk = flat[off['iegmn_original.att_mlp_key_ROT.0.weight']:]
            gq = flat[off['iegmn_original.att_mlp_query_ROT.0.weight']:]
            dh_cur, dh_nxt = ws.dh
            dx_cur, dx_nxt = ws.dx
            drop = fwd.get('dropout')   # the forward's masks, regenerated from its key (NULL: no dropout)
            dref = C.byref(drop.struct) if drop is not None else None
            nat.check(lib.eqd_bwd_head_dropout(g, C.byref(fwd['head'].struct), nat.ptr(fwd['h']), nat.ptr(fwd['x64']),
                                               nat.ptr(fwd['cov']), nat.ptr(fwd['x_lig_in']), nat.ptr(d_coors),
                                               nat.ptr(d_keypts), nat.ptr(d_rot), nat.ptr(d_trans), nat.ptr(ws.head_ws),
                                               ws.head_ws_bytes, nat.ptr(dh_cur), nat.ptr(dx_cur), nat.ptr(ws.dpre),
                                               nat.ptr(gk), nat.ptr(gq), dref, L, st), 'eqd_bwd_head')
            if capture is not None:
                capture.append({'head': True, 'dh': dh_cur.reshape(-1)[:N * 64].clone().view(N, 64), 'dx': dx_cur.clone()})
            hm = self.head_maps()
            nch = self._tn(ws, fwd['h'], 64, 64, ws.dpre, 64, 64, N, 1.0, True, st)
            self._reduce(ws.partial, nch, 64 * 64, hm['wm'], flat, st)
            self._reduce(ws.colsum, nch, 64, hm['bm'], flat, st)
            buckets = {lab: (lo, hi) for lab, lo, hi in lay_out.buckets}
            if on_bucket_done:
                on_bucket_done('head', *buckets['head'])
            so = fwd['stash_offsets']
            sbase = fwd['stash'].data_ptr()
            sp = lambda o: C.c_void_p(sbase + o)
            h0_ptr = sp(so[0])
            ws.dh0.zero_()
            done_modules = set()
            first_use = {}
            for li, lm in enumerate(iegmn.iegmn_layers):
                first_use.setdefault(id(lm), li)
            for li in reversed(range(L)):
                lm = iegmn.iegmn_layers[li]
                lp_obj: PackedLayer = fwd['layers'][li]
                tp = self.layer_pack(lm)
                lp = C.byref(lp_obj.struct)
                dh, dhp, pw = tp.dh, tp.dhp, tp.pw
                h_in = h0_ptr if li == 0 else sp(so[3] + li * so[4])
                ldh = nat.H0_PAD if li == 0 else nat.HID
                x_in = sp(so[1] + li * so[2])
                aggr, mu = sp(so[5] + li * so[6]), sp(so[7] + li * so[8])
                ldmu = nat.H0_PAD if dh == nat.H0 else nat.HID
                nat.check(lib.eqd_project(g, lp, h_in, ldh, nat.ptr(ws.proj), st), 'eqd_project')
                nparts = C.c_int32(0)
                nat.check(lib.eqd_bwd_node_mlp_dropout(g, lp, nat.ptr(tp.t['w_node1_lin']), nat.ptr(tp.t['w_node2_lin']),
                                                       h_in, ldh, aggr, mu, ldmu, h0_ptr, nat.ptr(dh_cur), nat.ptr(dh_nxt),
                                                       nat.ptr(ws.daggr), nat.ptr(ws.dmu), nat.ptr(ws.dh0), nat.ptr(ws.n5),
                                                       nat.ptr(ws.du), nat.ptr(ws.vec), C.byref(nparts), dref, li, st),
                          'eqd_bwd_node_mlp')
                self._reduce(ws.vec, nparts.value, 144, tp.maps['nodevec'], flat, st)
                # node MLP weight gradients
                sk = float(lp_obj.struct.dev.skip_weight_h) if dh == nat.HID else 1.0
                nch = self._tn(ws, ws.n5, dhp, dhp, dh_cur, 64, 64, N, sk, True, st)
                self._reduce(ws.partial, nch, dhp * 64, tp.maps['node2'], flat, st)
                self._reduce(ws.colsum, nch, 64, tp.maps['node2_bias'], flat, st)
                for name, X, ldx, K, want in (('node_h', h_in, ldh, dhp, True), ('node_aggr', aggr, 64, 64, False),
                                              ('node_mu', mu, ldmu, dhp, False), ('node_h0', h0_ptr, nat.H0_PAD, nat.H0_PAD, False)):
                    nchx = C.c_int32(0)
                    nat.check(lib.eqd_tn_gemm(X, ldx, K, nat.ptr(ws.du), dhp, dhp, N, 1.0, nat.ptr(ws.partial),
                                              nat.ptr(ws.colsum) if want else None, C.byref(nchx), st), 'eqd_tn_gemm')
                    self._reduce(ws.partial, nchx.value, K * dhp, tp.maps[name], flat, st)
                    if want:
                        self._reduce(ws.colsum, nchx.value, dhp, tp.maps['node1_bias'], flat, st)
                nat.check(lib.eqd_bwd_attention(g, lp, nat.ptr(ws.proj), mu, ldmu, nat.ptr(ws.dmu), nat.ptr(ws.dP),
                                                nat.ptr(ws.rowstat), st), 'eqd_bwd_attention')
                nat.check(lib.eqd_bwd_edge_dropout(g, lp, nat.ptr(tp.t['w2lin']), nat.ptr(tp.t['w3lin']), nat.ptr(ws.proj),
                                                   x_in, nat.ptr(ws.daggr), nat.ptr(dx_cur), nat.ptr(ws.ein), nat.ptr(ws.n1),
                                                   nat.ptr(ws.msg), nat.ptr(ws.dz3), nat.ptr(ws.dmsg), nat.ptr(ws.dz1),
                                                   nat.ptr(ws.dxrel), nat.ptr(ws.vec), C.byref(nparts), dref, li, st),
                          'eqd_bwd_edge')
                self._reduce(ws.vec, nparts.value, 256, tp.maps['edgevec'], flat, st)
                nch = self._tn(ws, ws.ein, 44, 44, ws.dz1, 64, 64, E, 1.0, False, st)
                self._reduce(ws.partial, nch, 44 * 64, tp.maps['edge1'], flat, st)
                nch = self._tn(ws, ws.n1, 64, 64, ws.dmsg, 64, 64, E, 1.0, True, st)
                self._reduce(ws.partial, nch, 64 * 64, tp.maps['edge2'], flat, st)
                self._reduce(ws.colsum, nch, 64, tp.maps['edge2_bias'], flat, st)
                nch = self._tn(ws, ws.msg, 64, 64, ws.dz3, 64, 64, E, 1.0, True, st)
                self._reduce(ws.partial, nch, 64 * 64, tp.maps['edge3'], flat, st)
                self._reduce(ws.colsum, nch, 64, tp.maps['edge3_bias'], flat, st)
                nat.check(lib.eqd_bwd_edge_gather(g, nat.ptr(ws.out_ptr), nat.ptr(ws.out_edge), nat.ptr(ws.dz1),
                                                  nat.ptr(ws.dxrel), nat.ptr(dx_cur), float(lp_obj.struct.dev.x_connection_init),
                                                  nat.ptr(ws.dP), pw, nat.ptr(dx_nxt), st), 'eqd_bwd_edge_gather')
                if capture is not None:
                    rows = lambda t, w, n=N: t.reshape(-1)[:n * w].clone().view(n, w)
                    capture.append({'layer': li, 'dh_part': rows(dh_nxt, dhp), 'daggr': ws.daggr.clone(), 'dmu': rows(ws.dmu, dhp),
                                    'dz1': ws.dz1[:E].clone(), 'dxrel': ws.dxrel[:E].clone(), 'dP': rows(ws.dP, pw),
                                    'dx': dx_nxt.clone(), 'dh0': ws.dh0.clone()})
                nat.check(lib.eqd_bwd_project(g, lp, nat.ptr(tp.t['w_projT']), nat.ptr(ws.dP), nat.ptr(dh_nxt), st),
                          'eqd_bwd_project')
                if capture is not None:
                    capture[-1]['dh'] = dh_nxt.reshape(-1)[:N * dhp].clone().view(N, dhp)
                nchx = C.c_int32(0)
                nat.check(lib.eqd_tn_gemm(h_in, ldh, dhp, nat.ptr(ws.dP), pw, pw, N, 1.0, nat.ptr(ws.partial),
                                          nat.ptr(ws.colsum), C.byref(nchx), st), 'eqd_tn_gemm')
                self._reduce(ws.partial, nchx.value, dhp * pw, tp.maps['proj'], flat, st)
                self._reduce(ws.colsum, nchx.value, pw, tp.maps['proj_bias'], flat, st)
                dh_cur, dh_nxt = dh_nxt, dh_cur
                dx_cur, dx_nxt = dx_nxt, dx_cur
                if on_bucket_done and first_use[id(lm)] == li:   # a shared module completes at its FIRST use
                    lab = lay_out.module_bucket[id(lm)]
                    on_bucket_done(lab, *buckets[lab])
            demb = flat[off['iegmn_original.residue_emb_layer.weight']:]
            nat.check(lib.eqd_bwd_embed(g, nat.ptr(fwd['res_l']), nat.ptr(fwd['res_r']), nat.ptr(ws.dh0), nat.ptr(dh_cur),
                                        nat.ptr(demb), st), 'eqd_bwd_embed')
            if on_bucket_done:
                on_bucket_done('emb', *buckets['emb'])
        return flat


class _HotPath(torch.autograd.Function):
    """autograd node of the whole hot path: forward = eqd_iegmn_forward with a stash, backward = the CUDA backward."""

    @staticmethod
    def forward(ctx, holder, *params):
        eng: TrainEngine = holder['engine']
        fwd = eng.forward(holder['graph'], holder.get('log'))
        holder['fwd'] = fwd
        ctx.holder = holder
        return fwd['ligand_coors'], fwd['keypts'], fwd['rotation'], fwd['translation']

    @staticmethod
    def backward(ctx, d_coors, d_keypts, d_rot, d_trans):
        holder = ctx.holder
        eng: TrainEngine = holder['engine']
        flat = eng.backward(holder['fwd'], d_coors, d_keypts, d_rot, d_trans)
        return (None, *eng.layout.views(flat))


def autograd_forward(model, graph, log=None):
    """Runs the model's hot path as ONE autograd node and returns (raw outputs dict, the four differentiable tensors)."""
    eng = getattr(model, '_eqd_train_engine', None)
    if eng is None or eng.device != model.iegmn_original.residue_emb_layer.weight.device:
        eng = TrainEngine(model)
        model._eqd_train_engine = eng
    holder = {'engine': eng, 'graph': graph, 'log': log}
    outs = _HotPath.apply(holder, *eng.layout.params)
    return holder['fwd'], outs


# ---- fused data-parallel training step -------------------------------------------------------------------------------

def allreduce_buckets(flat: torch.Tensor, buckets, world: int, group=None):
    """Sum-all-reduce of a flat gradient buffer bucket by bucket (same result as one all-reduce of the whole buffer:
    buckets are disjoint slices).  Host-side helper shared by the trainer and the gloo test."""
    if world <= 1:
        return
    import torch.distributed as dist
    for _, lo, hi in buckets:
        dist.all_reduce(flat[lo:hi], op=dist.ReduceOp.SUM, group=group)


class DataParallelTrainer:
    """One training step of the reference (src/train.py:88-169) on the engine, data-parallel over pairs:

        forward (stash) -> device losses (MSE + exact-EMD OT + intersection, losses.cu) -> CUDA backward into ONE flat
        fp32 gradient -> per-bucket NCCL all-reduce on a side stream, launched as soon as a bucket's last kernel is
        queued (head first: 49 % of the parameters; then the layers last to first) so that it overlaps the rest of the
        backward -> global-norm partials -> fused clip_grad_norm_ + Adam on the flat parameter buffer.

    Each rank normalises its loss by its LOCAL pair count (train.py:143-146); gradients are averaged over ranks, which is
    the reference's global-batch mean when ranks hold equally many pairs.  The model's parameters are re-pointed at
    slices of one flat buffer (``param.data`` views), so the update is a single kernel and the all-reduce needs no
    packing."""

    def __init__(self, model, lr: float, weight_decay: float = 0.0, clip: float = 100.0, betas=(0.9, 0.999), eps: float = 1e-8,
                 pocket_ot_loss_weight: float = 1.0, intersection_loss_weight: float = 10.0, intersection_sigma: float = 25.0,
                 intersection_surface_ct: float = 10.0, world: int = 1, group=None):
        self.model = model.train()
        self.engine = TrainEngine(model)
        self.layout = self.engine.layout
        dev = self.engine.device
        self.device, self.world, self.group = dev, int(world), group
        self.flat_w = torch.empty(self.layout.total, dtype=_f32, device=dev)
        with torch.no_grad():
            for p, v in zip(self.layout.params, self.layout.views(self.flat_w)):
                v.copy_(p.detach().to(_f32))
                p.data = v                                       # parameters now live in the flat buffer
        self.m = torch.zeros_like(self.flat_w)
        self.v = torch.zeros_like(self.flat_w)
        self.flat_g = torch.zeros_like(self.flat_w)
        self.sq = torch.empty(256, dtype=torch.float64, device=dev)
        self.norm = torch.zeros(1, dtype=_f32, device=dev)
        self.hp = dict(lr=float(lr), wd=float(weight_decay), clip=float(clip), b1=float(betas[0]), b2=float(betas[1]), eps=float(eps))
        self.loss_args = (pocket_ot_loss_weight, intersection_loss_weight, intersection_sigma, intersection_surface_ct)
        self.steps = 0
        self.comm = torch.cuda.Stream(dev) if self.world > 1 else None
        self.rank = 0
        if self.world > 1:
            import torch.distributed as dist
            self.rank = dist.get_rank(group)
        self.engine.rank = self.rank   # equally seeded ranks draw different dropout masks
        self.lib = nat.load()

    def invalidate_packed(self):
        for lay in self.model.iegmn_original.iegmn_layers:
            lay._packed = None
        self.model.iegmn_original._head = None
        self.engine._packs.clear()

    def step(self, graph, targets) -> Dict:
        from .losses import device_losses
        dev, eng = self.device, self.engine
        with torch.cuda.device(dev):
            compute = torch.cuda.current_stream(dev)
            fwd = eng.forward(graph, self.model.log)
            res = device_losses(fwd['plan'], fwd['ligand_coors'], fwd['keypts'], targets, *self.loss_args)
            self.flat_g.zero_()                                  # optimizer.zero_grad() (train.py:88)

            def bucket_done(label, lo, hi):
                if self.world <= 1:
                    return
                import torch.distributed as dist
                ev = torch.cuda.Event()
                ev.record(compute)
                with torch.cuda.stream(self.comm):
                    self.comm.wait_event(ev)
                    dist.all_reduce(self.flat_g[lo:hi], op=dist.ReduceOp.SUM, group=self.group)

            eng.backward(fwd, res['dcoors'], res['dkeypts'], flat=self.flat_g, on_bucket_done=bucket_done)
            if self.world > 1:
                compute.wait_stream(self.comm)
            st = C.c_void_p(compute.cuda_stream)
            self.steps += 1
            nat.check(self.lib.eqd_sqnorm_partials(nat.ptr(self.flat_g), self.layout.total, nat.ptr(self.sq), 256, st), 'eqd_sqnorm_partials')
            h = self.hp
            nat.check(self.lib.eqd_clip_adam(nat.ptr(self.flat_w), nat.ptr(self.flat_g), nat.ptr(self.m), nat.ptr(self.v),
                                             self.layout.total, nat.ptr(self.sq), 256, h['clip'], h['lr'], h['b1'], h['b2'], h['eps'],
                                             h['wd'], self.steps, 1.0 / self.world, nat.ptr(self.norm), st), 'eqd_clip_adam')
            self.invalidate_packed()
        return {'loss': res['total'], 'grad_norm': self.norm, 'err': res['err'], 'fwd': fwd, 'parts': res['parts']}
