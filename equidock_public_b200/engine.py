"""Host side of the B200 IEGMN forward engine: weight repacking, batch topology ("plan"), buffer
management and kernel sequencing over the C ABI (``include/eqd_iegmn.h``).

PyTorch is used for device memory, streams and a few index-building ops only; all arithmetic of
the hot path runs in the hand-written sm_100a kernels of ``csrc/``.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import sys
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _native as nat
from .hetero_graph import LIGAND, LL, RECEPTOR, RR


def _dev_f32(t, device):
    return t.detach().to(device=device, dtype=torch.float32).contiguous()


def _host_f32(t):
    return t.detach().to(device='cpu', dtype=torch.float32).contiguous()


def _upload_blob(tensors: Dict[str, torch.Tensor], device) -> Dict[str, torch.Tensor]:
    """Packs host tensors (fp32 / bf16) into ONE 256-byte-aligned byte blob, uploads it with a single H2D copy and
    returns device views.  All weight repacking happens on the host: the only GPU work of a (re)pack is one memcpy, so
    no ATen kernel of a repack ever appears among the engine's kernels."""
    offs, total = {}, 0
    for k, t in tensors.items():
        offs[k] = total
        total += (t.numel() * t.element_size() + 255) & ~255
    host = torch.zeros(max(total, 256), dtype=torch.uint8)
    for k, t in tensors.items():
        n = t.numel() * t.element_size()
        host[offs[k]:offs[k] + n] = t.contiguous().view(-1).view(torch.uint8)
    dev = host.to(device)
    out = {}
    for k, t in tensors.items():
        n = t.numel() * t.element_size()
        out[k] = dev[offs[k]:offs[k] + n].view(t.dtype).view(t.shape)
    out['_blob'] = dev
    return out


def umma_bf16x3(w: torch.Tensor) -> torch.Tensor:
    """[N][K] fp32 weight (nn.Linear layout, K % 8 == 0) -> 3 bf16 splits (w ~ w0+w1+w2, round to nearest), each in
    the UMMA canonical K-major no-swizzle layout: element (n,k) at (k/8)*N*16 + (n/8)*128 + (n%8)*16 + (k%8)*2 bytes.
    Returns a flat bf16 tensor [3 * N * K]."""
    n, k = w.shape
    assert n % 8 == 0 and k % 8 == 0
    parts, r = [], w.to(torch.float32)
    for _ in range(3):
        b = r.to(torch.bfloat16)
        parts.append(b)
        r = r - b.to(torch.float32)
    out = [b.reshape(n // 8, 8, k // 8, 8).permute(2, 0, 1, 3).contiguous().reshape(-1) for b in parts]
    return torch.cat(out)


# EQD_LAYER0_FFMA=1 keeps the 69-wide layer 0 on the fp32 CUDA-core kernels (A/B comparisons)
_LAYER0_FFMA = bool(int(__import__('os').environ.get('EQD_LAYER0_FFMA', '0')))
# EQD_PY_FORWARD=1: drive the stages one C call at a time from Python instead of through eqd_iegmn_forward
_PY_FORWARD = bool(int(__import__('os').environ.get('EQD_PY_FORWARD', '0')))


class PackedLayer:
    """One IEGMN_Layer's parameters repacked k-major for the kernels (see eqd_layer_params)."""

    def __init__(self, sd: Dict[str, torch.Tensor], device, skip_weight_h: float, x_connection_init: float,
                 leaky_slope: float):
        f = lambda k: _host_f32(sd[k])      # everything below is host arithmetic; ONE upload at the end
        w1, b1 = f('edge_mlp.0.weight'), f('edge_mlp.0.bias')
        wq, wk, wv = f('att_mlp_Q.0.weight'), f('att_mlp_K.0.weight'), f('att_mlp_V.0.weight')
        w5, b5 = f('node_mlp.0.weight'), f('node_mlp.0.bias')
        w6, b6 = f('node_mlp.4.weight'), f('node_mlp.4.bias')
        dh = int(wq.shape[0])
        if dh not in (nat.HID, nat.H0):
            raise ValueError(f'IEGMN layer width {dh} is not supported by the CUDA engine (64 or 69)')
        dhp = nat.HID if dh == nat.HID else nat.H0_PAD
        n_e = nat.EDGE_FEATS + nat.N_RBF
        assert w1.shape == (nat.HID, 2 * dh + n_e) and w5.shape == (dh, 2 * dh + nat.HID + nat.H0)
        z = lambda *s: torch.zeros(*s, dtype=torch.float32)
        pw = 128 + 3 * dhp
        w_proj, b_proj = z(dhp, pw), z(pw)
        w_proj[:dh, 0:64] = w1[:, 0:dh].t()
        w_proj[:dh, 64:128] = w1[:, dh:2 * dh].t()
        w_proj[:dh, 128:128 + dh] = wq.t()
        w_proj[:dh, 128 + dhp:128 + dhp + dh] = wk.t()
        w_proj[:dh, 128 + 2 * dhp:128 + 2 * dhp + dh] = wv.t()
        b_proj[64:128] = b1
        w_edge1 = z(44, 64)
        w_edge1[:n_e] = w1[:, 2 * dh:].t()
        w_node1 = z(2 * dhp + 64 + nat.H0_PAD, dhp)
        w_node1[0:dh, :dh] = w5[:, 0:dh].t()
        w_node1[dhp:dhp + 64, :dh] = w5[:, dh:dh + 64].t()
        w_node1[dhp + 64:dhp + 64 + dh, :dh] = w5[:, dh + 64:2 * dh + 64].t()
        w_node1[2 * dhp + 64:2 * dhp + 64 + nat.H0, :dh] = w5[:, 2 * dh + 64:].t()
        pad = lambda v: torch.cat([v, z(dhp - dh)]) if dhp > dh else v.clone()
        w_node2 = z(dhp, 64)
        w_node2[:dh] = w6.t()
        self.dh, self.dhp = dh, dhp
        w1e = z(64, 48)
        w1e[:, :n_e] = w1[:, 2 * dh:]
        # coors_mlp.0 applied to msg = W2 a1 + b2 is linear in a1: (W3 W2) a1 + (W3 b2 + b3); the tensor-core edge stage
        # evaluates [W2 ; W3 W2] as one N=128 panel on the same A operand (folded in fp64, stored fp32 -> bf16x3)
        w2d, w3d = f('edge_mlp.4.weight').double(), f('coors_mlp.0.weight').double()
        w32 = (w3d @ w2d).float()
        b32 = (w3d @ f('edge_mlp.4.bias').double() + f('coors_mlp.0.bias').double()).float()
        w_edge_tc = torch.cat([umma_bf16x3(w1e), umma_bf16x3(torch.cat([f('edge_mlp.4.weight'), w32]))]).contiguous()
        assert w_edge_tc.numel() * 2 == 67584
        self.edge_consts_host = torch.stack([f('edge_mlp.3.weight'), f('edge_mlp.3.bias'), f('edge_mlp.4.bias'),
                                             b32, f('coors_mlp.4.weight').reshape(-1)]).cpu().contiguous()
        tc = {}
        self.node_consts_host = self.proj_bias_host = None
        if dh == nat.HID:  # tensor-core node stage panels (64-wide layers)
            w5p = z(64, 272)
            w5p[:, :261] = w5
            tc['w_node_tc'] = torch.cat([umma_bf16x3(w5p), umma_bf16x3(w6)]).contiguous()
            groups = [w1[:, 0:64], w1[:, 64:128], wq, wk, wv]
            tc['w_proj_tc'] = torch.cat([umma_bf16x3(gw.contiguous()) for gw in groups]).contiguous()
            assert tc['w_node_tc'].numel() * 2 == 129024 and tc['w_proj_tc'].numel() * 2 == 122880
            self.node_consts_host = torch.stack([b5, f('node_mlp.3.weight'), f('node_mlp.3.bias'), b6]).cpu().contiguous()
            self.proj_bias_host = b_proj.cpu().contiguous()
        else:  # layer 0 (69 wide, h = h0): K padded to 80; channels 64..68 of Q / K / V form a sixth N = 16 group
            p80 = lambda w: torch.cat([w, z(w.shape[0], 80 - w.shape[1])], 1)
            x16 = z(16, 69)
            x16[0:4], x16[4:8], x16[8], x16[9], x16[10:15] = wk[64:68], wv[64:68], wk[68], wv[68], wq[64:69]
            groups = [w1[:, 0:69], w1[:, 69:138], wq[0:64], wk[0:64], wv[0:64], x16]
            tc['w_proj_tc'] = torch.cat([umma_bf16x3(p80(gw).contiguous()) for gw in groups]).contiguous()
            w5p = z(80, 224)   # [h0 (h and h0 blocks folded, 80) | aggr (64) | mu (80)]
            w5p[:69, 0:69] = (w5[:, 0:69].double() + w5[:, 202:271].double()).float()
            w5p[:69, 80:144] = w5[:, 69:133]
            w5p[:69, 144:213] = w5[:, 133:202]
            tc['w_node_tc'] = torch.cat([umma_bf16x3(w5p), umma_bf16x3(p80(w6).contiguous())]).contiguous()
            assert tc['w_proj_tc'].numel() * 2 == 161280 and tc['w_node_tc'].numel() * 2 == 138240
            p80v = lambda v: torch.cat([v, z(80 - v.shape[0])])
            self.node_consts_host = torch.cat([p80v(b5), p80v(f('node_mlp.3.weight')), p80v(f('node_mlp.3.bias')), b6]).cpu().contiguous()
            pb = z(320)
            pb[64:128] = b1
            self.proj_bias_host = pb.cpu().contiguous()
        self.t = _upload_blob({
            **tc,
            'w_proj': w_proj, 'b_proj': b_proj, 'w_edge1': w_edge1,
            'edge_ln_g': f('edge_mlp.3.weight'), 'edge_ln_b': f('edge_mlp.3.bias'),
            'w_edge2': f('edge_mlp.4.weight').t().contiguous(), 'b_edge2': f('edge_mlp.4.bias'),
            'w_coor1': f('coors_mlp.0.weight').t().contiguous(), 'b_coor1': f('coors_mlp.0.bias'),
            'w_coor2': f('coors_mlp.4.weight').reshape(-1).contiguous(),
            'w_node1': w_node1, 'b_node1': pad(b5),
            'node_ln_g': pad(f('node_mlp.3.weight')), 'node_ln_b': pad(f('node_mlp.3.bias')),
            'w_node2': w_node2, 'b_node2': b6, 'w_edge_tc': w_edge_tc,
        }, device)
        lay = nat.EqdLayer()
        s = lay.dev
        s.dh, s.dhp = dh, dhp
        for k, v in self.t.items():
            if not k.startswith('_'):
                setattr(s, k, v.data_ptr())
        for name, host in (('edge', self.edge_consts_host), ('node', self.node_consts_host), ('proj_bias', self.proj_bias_host)):
            if host is not None:   # host VALUES, copied into the descriptor (the kernels get them as launch constants)
                flat = host.reshape(-1).numpy()
                C.memmove(C.addressof(getattr(lay.consts, name)), flat.ctypes.data, flat.nbytes)
        s.b_coor2 = float(sd['coors_mlp.4.bias'].detach().reshape(-1)[0].item())
        s.skip_weight_h, s.x_connection_init, s.leaky_slope = skip_weight_h, x_connection_init, leaky_slope
        self.struct = lay


class PackedHead:
    """Head parameters for the kernels.  mlp_h_mean_ROT's weight is needed k-major (transposed, 64 x 64: one tiny copy); the
    3200 x 64 key / query projections and the bias are used IN PLACE when they already are fp32, contiguous, 16-byte
    aligned device tensors (the normal case: no 1.6 MB round trip through the host per parameter version), else
    through one host-packed upload."""

    def __init__(self, w_mean, b_mean, w_key, w_query, device, leaky_slope: float):
        dev = torch.device(device)
        inplace = all(t.is_cuda and t.device == dev and t.dtype == torch.float32 and t.is_contiguous() and t.data_ptr() % 16 == 0
                      for t in (b_mean, w_key, w_query)) and w_mean.is_cuda
        if inplace:
            self.t = {'w_mean': w_mean.detach().to(torch.float32).t().contiguous(), 'b_mean': b_mean.detach(),
                      'w_key': w_key.detach(), 'w_query': w_query.detach()}
        else:
            self.t = _upload_blob({'w_mean': _host_f32(w_mean).t().contiguous(), 'b_mean': _host_f32(b_mean),
                                   'w_key': _host_f32(w_key), 'w_query': _host_f32(w_query)}, device)
        assert self.t['w_key'].shape == (nat.HEADS * nat.HID, nat.HID)
        s = nat.EqdHeadParams()
        for k, v in self.t.items():
            if not k.startswith('_'):
                setattr(s, k, v.data_ptr())
        s.leaky_slope = leaky_slope
        self.struct = s
        # weights-only fold of the 50-head key / query projections (eqd_head_fold), done once per parameter version on the device
        self.m_qk = torch.empty(nat.HEADS, nat.HID, nat.HID, dtype=torch.float64, device=device)
        with torch.cuda.device(device):
            nat.check(nat.load().eqd_head_fold(C.byref(s), self.m_qk.data_ptr(), torch.cuda.current_stream().cuda_stream),
                      'eqd_head_fold')
        s.m_qk = self.m_qk.data_ptr()


def _aligned_he(he, device):
    """The edge-feature matrix as the edge kernels need it: fp32, contiguous, 16-byte aligned base and readable up to the
    next 16-byte boundary past its end (TMA bulk copies over-read the last row).  A caller's tensor that already satisfies
    this is used in place (no copy of the largest input); row slices of a batched ``he`` (``dgl.unbatch`` /
    ``hetero_graph.unbatch``: offset = first_edge * 108 bytes) generally do not and are copied into an owned, padded
    buffer."""
    he = he.to(device=device, dtype=torch.float32).contiguous()
    nbytes = he.numel() * 4
    try:
        room = he.untyped_storage().nbytes() - he.storage_offset() * 4
    except RuntimeError:
        room = nbytes
    if he.data_ptr() % 16 == 0 and room >= ((nbytes + 15) & ~15):
        return he
    buf = torch.empty(((nbytes + 15) // 16) * 4 + 4, dtype=torch.float32, device=device)
    own = buf[:he.numel()].view(he.shape)
    own.copy_(he)
    return own


class GraphPlan:
    """Batch topology in the engine's layout (see the numbering comment in eqd_iegmn.h)."""

    def __init__(self, n_lig: Sequence[int], n_rec: Sequence[int], src_l, dst_l, src_r, dst_r, he_l, he_r,
                 device, max_in_degree: int = 10):
        n_lig = [int(v) for v in n_lig]
        n_rec = [int(v) for v in n_rec]
        assert len(n_lig) == len(n_rec) and len(n_lig) > 0
        self.n_pairs = len(n_lig)
        self.forward_ws_bytes = None   # eqd_forward_workspace_bytes(), filled on first use
        self.n_lig_list, self.n_rec_list = n_lig, n_rec
        self.N_l, self.N_r = sum(n_lig), sum(n_rec)
        self.N = self.N_l + self.N_r
        self.device = device
        i32 = dict(dtype=torch.int32, device=device)
        src_l, dst_l = src_l.to(**i32), dst_l.to(**i32)
        src_r, dst_r = src_r.to(**i32), dst_r.to(**i32)
        self.E_l, self.E_r = int(src_l.shape[0]), int(src_r.shape[0])
        self.E = self.E_l + self.E_r
        self.col_src = torch.cat([src_l, src_r + self.N_l]).contiguous()
        self.edge_dst = torch.cat([dst_l, dst_r + self.N_l]).contiguous()
        # CSR by destination; the kernels assume edges arrive grouped by ascending destination
        # (protein_utils.py:339-346 emits them that way).  `unsorted` stays on the device and is
        # read together with the per-pair status (one sync per forward).
        d64 = self.edge_dst.long()
        self.unsorted = ((d64[1:] < d64[:-1]).any() if self.E > 1 else torch.zeros((), dtype=torch.bool, device=device))
        self.unsorted_i32 = self.unsorted.to(torch.int32).reshape(1)
        self._arange = None
        # row_ptr[n] = first edge whose destination is >= n.  searchsorted on the (sorted) destination list needs no
        # host sync -- torch.bincount would block the CPU on the previous batch and break the copy/compute overlap.
        self.row_ptr = torch.searchsorted(self.edge_dst, torch.arange(self.N + 1, **i32), out_int32=True).contiguous()
        self.he_l, self.he_r = _aligned_he(he_l, device), _aligned_he(he_r, device)
        assert self.he_l.shape == (self.E_l, nat.EDGE_FEATS) and self.he_r.shape == (self.E_r, nat.EDGE_FEATS)
        seg = np.zeros(2 * self.n_pairs + 1, dtype=np.int64)
        seg[1:] = np.cumsum(np.asarray(n_lig + n_rec, dtype=np.int64))
        tiles = []
        for s in range(2 * self.n_pairs):
            for n0 in range(int(seg[s]), int(seg[s + 1]), nat.TILE_ROWS):
                tiles.append((s, n0))
        self.seg_ptr_host = seg
        self.n_node_tiles = len(tiles)
        small = torch.from_numpy(np.concatenate([seg.astype(np.int32),
                                                 np.asarray(tiles, dtype=np.int32).reshape(-1)]))
        small = small.to(device, non_blocking=True)
        self.seg_ptr = small[:2 * self.n_pairs + 1]
        self.node_tiles = small[2 * self.n_pairs + 1:]
        self._small = small
        g = nat.EqdGraph()
        g.n_pairs, g.n_nodes, g.n_lig_nodes = self.n_pairs, self.N, self.N_l
        g.n_edges, g.n_lig_edges, g.max_in_degree = self.E, self.E_l, int(max_in_degree)
        g.seg_ptr, g.row_ptr = self.seg_ptr.data_ptr(), self.row_ptr.data_ptr()
        g.col_src, g.edge_dst = self.col_src.data_ptr(), self.edge_dst.data_ptr()
        g.he_lig, g.he_rec = self.he_l.data_ptr(), self.he_r.data_ptr()
        g.n_node_tiles, g.node_tiles = self.n_node_tiles, self.node_tiles.data_ptr()
        self.struct = g

    def refresh(self, graph) -> bool:
        """Re-derives the topology arrays IN PLACE from a graph object whose tensors were overwritten with a new batch
        of the same shape signature (same per-pair node counts and edge totals): every device pointer of the plan stays
        valid, which is what a captured CUDA graph of the forward needs.  Returns False when the shapes differ (the
        caller must build a new plan).  A handful of index ops on the current stream, no host sync."""
        n_l = [int(v) for v in graph.batch_num_nodes(LIGAND).tolist()]
        n_r = [int(v) for v in graph.batch_num_nodes(RECEPTOR).tolist()]
        src_l, dst_l = graph.edges(etype=LL)
        src_r, dst_r = graph.edges(etype=RR)
        if (n_l != self.n_lig_list or n_r != self.n_rec_list or int(src_l.shape[0]) != self.E_l
                or int(src_r.shape[0]) != self.E_r):
            return False
        E_l = self.E_l
        self.col_src[:E_l].copy_(src_l)
        torch.add(src_r, self.N_l, out=self.col_src[E_l:])
        self.edge_dst[:E_l].copy_(dst_l)
        torch.add(dst_r, self.N_l, out=self.edge_dst[E_l:])
        if self.E > 1:
            torch.any(self.edge_dst[1:] < self.edge_dst[:-1], dim=0, keepdim=True, out=self.unsorted.view(1))
        self.unsorted_i32.copy_(self.unsorted.view(1))
        if self._arange is None:
            self._arange = torch.arange(self.N + 1, dtype=torch.int32, device=self.device)
        torch.searchsorted(self.edge_dst, self._arange, out_int32=True, out=self.row_ptr)
        for own, new in ((self.he_l, graph.edges[LL].data['he']), (self.he_r, graph.edges[RR].data['he'])):
            if own.data_ptr() != new.data_ptr():
                own.copy_(new)
        return True

    @classmethod
    def from_graph(cls, graph, device, max_in_degree: int = 10) -> 'GraphPlan':
        """From a batched DGL heterograph (train_utils.py:61-100) or a ``PairGraphBatch``."""
        n_l = graph.batch_num_nodes(LIGAND).tolist()
        n_r = graph.batch_num_nodes(RECEPTOR).tolist()
        src_l, dst_l = graph.edges(etype=LL)
        src_r, dst_r = graph.edges(etype=RR)
        return cls(n_l, n_r, src_l, dst_l, src_r, dst_r, graph.edges[LL].data['he'], graph.edges[RR].data['he'],
                   device, max_in_degree)


def _sorted_copy(plan_args):
    """Slow path for graphs whose edges are not grouped by destination: stable sort + permute."""
    n_l, n_r, src_l, dst_l, src_r, dst_r, he_l, he_r, device, mid = plan_args
    out = []
    for s, d, he in ((src_l, dst_l, he_l), (src_r, dst_r, he_r)):
        perm = torch.sort(d.long(), stable=True).indices
        out.append((s[perm], d[perm], he[perm]))
    (sl, dl, hl), (sr, dr, hr) = out
    return n_l, n_r, sl, dl, sr, dr, hl, hr, device, mid


class _StatusPool:
    """Pinned int32 buffers for the per-forward status words, owned by exactly one pending forward at a time: taken from
    a free list by ``forward`` and handed back by ``resolve_status`` (or by the garbage collector if a caller drops an
    unresolved handle), so any number of forwards may be in flight without one overwriting another's flags.  Allocating
    page-locked memory per call (cudaHostAlloc) would stall the CPU for tens of milliseconds every few steps."""

    def __init__(self):
        import threading
        self.free, self.lock = [], threading.Lock()

    def take(self, n: int) -> torch.Tensor:
        with self.lock:
            for i, b in enumerate(self.free):
                if b.numel() >= n:
                    return self.free.pop(i)
        return torch.empty(max(n, 1024), dtype=torch.int32, pin_memory=True)

    def give(self, buf: torch.Tensor):
        with self.lock:
            if len(self.free) < 64:
                self.free.append(buf)


_STATUS_POOL = _StatusPool()


class _StatusLease:
    """Returns its pinned buffer to the pool when released (explicitly after the status was read, or on GC)."""

    def __init__(self, n):
        self.buf, self.n = _STATUS_POOL.take(n), n

    def view(self):
        return self.buf[:self.n]

    def release(self):
        if self.buf is not None:
            _STATUS_POOL.give(self.buf)
            self.buf = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class NativeStageTimer:
    """CUDA events recorded by eqd_iegmn_forward around every edge / node stage (io.stage_events), on the launching
    stream; in the Python driver the same handles are recorded through begin() / end()."""

    def __init__(self):
        self.lib, self.sets, self.spare = nat.load(), [], []

    def reserve(self, n_forwards, n_layers):
        """Creates the events of `n_forwards` forwards up front, so that a timed loop creates none."""
        for _ in range(n_forwards):
            self.spare.append((C.c_void_p * (4 * n_layers))(*[self.lib.eqd_event_create() for _ in range(4 * n_layers)]))

    def new_forward(self, n_layers):
        if self.spare and len(self.spare[-1]) == 4 * n_layers:
            arr = self.spare.pop()
        else:
            arr = (C.c_void_p * (4 * n_layers))(*[self.lib.eqd_event_create() for _ in range(4 * n_layers)])
        self.sets.append(arr)
        return arr

    def _pairs(self, name):
        off = 0 if name == 'edge_stage' else 2
        for arr in self.sets:
            for li in range(len(arr) // 4):
                yield arr[li * 4 + off], arr[li * 4 + off + 1]

    def mean_ms(self, name):
        v = [self.lib.eqd_event_elapsed_ms(a, b) for a, b in self._pairs(name)]
        v = [x for x in v if x >= 0]
        return float(np.mean(v)) if v else None

    def total_ms(self, name):
        return float(sum(x for x in (self.lib.eqd_event_elapsed_ms(a, b) for a, b in self._pairs(name)) if x >= 0))

    def close(self):
        for arr in self.sets + self.spare:
            for e in arr:
                self.lib.eqd_event_destroy(e)
        self.sets, self.spare = [], []


class IEGMNEngine:
    """Runs the IEGMN stack + keypoints + Kabsch for one plan on the current CUDA stream."""

    @staticmethod
    def launches_per_forward(n_layers: int) -> int:
        """Kernels of csrc/ launched by one forward: embed, project (layer 0), per layer edge stage + node stage
        (attention, node MLP, next layer's projections), then head_mean, tile_ptr, head_qbar, head_u, keypoints,
        keypoint_cov, kabsch_apply."""
        n = 2 + 7
        for li in range(n_layers):
            last = li == n_layers - 1
            n += 1 + 2 + (0 if last else 1)
        return n

    def __init__(self, device):
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise nat.NativeLibraryError('the IEGMN engine runs on a CUDA device only (no CPU fallback)')
        self.lib = nat.load()

    def forward(self, plan: GraphPlan, emb: torch.Tensor, layers: List[PackedLayer], head: PackedHead,
                res_l, res_r, mu_l, mu_r, x_l, x_r, check_status: bool = True, log=None,
                stage_timer=None, record_event: bool = True, train_stash=None, dropout_p: float = 0.0,
                dropout_rank: int = 0) -> Dict[str, torch.Tensor]:
        """One forward = ONE call into the library (eqd_iegmn_forward): the per-stage entry points are chained in C on
        the current stream out of a single workspace allocation.  EQD_PY_FORWARD=1 selects the stage-by-stage Python
        driver below instead (same kernels; used to A/B the two and by the per-stage tests).

        ``dropout_p`` > 0 (training): a fresh 64-bit key is drawn on the device for this call (``nat.Dropout``) and the
        forward applies the four dropout sites (eqd_iegmn_forward_dropout); the key travels in ``out['dropout']`` so that the
        backward regenerates the same masks.  ``dropout_rank`` separates the masks of data-parallel ranks."""
        with torch.cuda.device(self.device):   # the raw launches below go to the CURRENT device: make it the model's
            drop = nat.Dropout(dropout_p, self.device, dropout_rank) if dropout_p > 0 else None
            if _PY_FORWARD:
                if drop is not None:
                    raise NotImplementedError('dropout runs through eqd_iegmn_forward_dropout only (unset EQD_PY_FORWARD)')
                return self._forward_py(plan, emb, layers, head, res_l, res_r, mu_l, mu_r, x_l, x_r, check_status, log,
                                        stage_timer)
            return self._forward_native(plan, emb, layers, head, res_l, res_r, mu_l, mu_r, x_l, x_r, check_status, log,
                                        stage_timer, record_event, train_stash, drop)

    def _forward_native(self, plan, emb, layers, head, res_l, res_r, mu_l, mu_r, x_l, x_r, check_status, log,
                        stage_timer, record_event=True, train_stash=None, drop=None):
        lib, dev = self.lib, self.device
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        N, B = plan.N, plan.n_pairs
        f32 = dict(dtype=torch.float32, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        cf = lambda t: t.to(**f32).contiguous()
        res_l, res_r, mu_l, mu_r, x_l, x_r = map(cf, (res_l, res_r, mu_l, mu_r, x_l, x_r))
        assert x_l.shape == (plan.N_l, 3) and x_r.shape == (plan.N_r, 3)
        g = C.byref(plan.struct)
        if plan.forward_ws_bytes is None:
            plan.forward_ws_bytes = int(lib.eqd_forward_workspace_bytes(g))
        ws = torch.empty(plan.forward_ws_bytes, dtype=torch.uint8, device=dev)
        # outputs (separate allocations: the kernels assume 16-byte aligned rows)
        rot, trans = torch.empty(B, 3, 3, **f32), torch.empty(B, 1, 3, **f32)
        lig_out, h_fin = torch.empty(plan.N_l, 3, **f32), torch.empty(N, nat.HID, **f32)
        sing, x_fin = torch.empty(B, 3, **f64), torch.empty(N, 3, **f64)
        keyp, cov, ymean = torch.empty(2 * B, nat.HEADS, 3, **f64), torch.empty(B, 9, **f64), torch.empty(2 * B, 3, **f64)
        status = torch.empty(B + 1, dtype=torch.int32, device=dev)
        io = nat.EqdForwardIO()
        for name, t in (('emb', emb), ('res_lig', res_l), ('res_rec', res_r), ('mu_lig', mu_l), ('mu_rec', mu_r),
                        ('x_lig', x_l), ('x_rec', x_r), ('rot', rot), ('trans', trans), ('ligand_out', lig_out),
                        ('sing', sing), ('status', status), ('h_out', h_fin), ('x_out', x_fin), ('keypts', keyp),
                        ('cov', cov), ('ymean', ymean)):
            setattr(io, name, t.data_ptr())
        io.layer0_fp32 = 1 if _LAYER0_FFMA else 0
        if train_stash is not None:   # training: keep every layer's inputs for the backward kernels
            io.train_stash, io.train_stash_bytes = train_stash.data_ptr(), int(train_stash.numel())
        events = stage_timer.new_forward(len(layers)) if stage_timer is not None else None
        io.stage_events = C.cast(events, C.c_void_p) if events is not None else None
        larr = (C.POINTER(nat.EqdLayer) * len(layers))(*[C.pointer(l.struct) for l in layers])
        if drop is None:
            nat.check(lib.eqd_iegmn_forward(g, larr, len(layers), C.byref(head.struct), C.byref(io), nat.ptr(ws),
                                            plan.forward_ws_bytes, st), 'eqd_iegmn_forward')
        else:
            nat.check(lib.eqd_iegmn_forward_dropout(g, larr, len(layers), C.byref(head.struct), C.byref(io),
                                                    C.byref(drop.struct), nat.ptr(ws), plan.forward_ws_bytes, st),
                      'eqd_iegmn_forward_dropout')
        kab = lambda mask: nat.check(lib.eqd_kabsch_apply(
            g, nat.ptr(cov), nat.ptr(ymean), nat.ptr(x_l), nat.ptr(mask), nat.ptr(rot), nat.ptr(trans),
            nat.ptr(lig_out), nat.ptr(sing), nat.ptr(status), st), 'eqd_kabsch_apply')
        lease = _StatusLease(B + 2)
        status_host = lease.view()
        status_host[:B + 1].copy_(status, non_blocking=True)
        status_host[B + 1:].copy_(plan.unsorted_i32, non_blocking=True)
        status_event = None
        if record_event:     # (a CUDA-graph capture records its own event after every replay instead)
            status_event = torch.cuda.Event()
            status_event.record()
        out = {'status_lease': lease, 'ligand_coors': lig_out, 'keypts': keyp, 'rotation': rot, 'translation': trans,
               'h': h_fin, 'x64': x_fin, 'cov': cov, 'sing': sing, 'status': status, 'unsorted': plan.unsorted,
               'kabsch': kab, 'status_host': status_host, 'status_event': status_event, '_keep': (ws, ymean, x_l),
               'dropout': drop}
        if check_status:
            self.resolve_status(plan, out, kab, log)
        return out

    def _forward_py(self, plan: GraphPlan, emb: torch.Tensor, layers: List[PackedLayer], head: PackedHead,
                    res_l, res_r, mu_l, mu_r, x_l, x_r, check_status: bool = True, log=None,
                    stage_timer=None) -> Dict[str, torch.Tensor]:
        lib, dev = self.lib, self.device
        g = C.byref(plan.struct)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        N, B = plan.N, plan.n_pairs
        f32 = dict(dtype=torch.float32, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        cf = lambda t: t.to(**f32).contiguous()
        res_l, res_r, mu_l, mu_r, x_l, x_r = map(cf, (res_l, res_r, mu_l, mu_r, x_l, x_r))
        assert x_l.shape == (plan.N_l, 3) and x_r.shape == (plan.N_r, 3)
        h0 = torch.empty(N, nat.H0_PAD, **f32)
        x0 = torch.empty(N, 3, **f64)
        xa, xb = torch.empty(N, 3, **f64), torch.empty(N, 3, **f64)
        ha, hb = torch.empty(N, nat.HID, **f32), torch.empty(N, nat.HID, **f32)
        pa, pb = torch.empty(N, 128 + 3 * nat.H0_PAD, **f32), torch.empty(N, 128 + 3 * nat.H0_PAD, **f32)
        aggr = torch.empty(N, nat.HID, **f32)
        status = torch.zeros(B + 1, dtype=torch.int32, device=dev)
        mu = torch.empty(N, nat.HID, **f32)
        kv_bytes = lib.eqd_kv_blocks_bytes(N)
        kv = torch.empty(kv_bytes, dtype=torch.uint8, device=dev)
        # rows never written (tail of the last 8-node block + the 8 pad blocks of each (K|V, split) plane) reach
        # the P.V MMA as 0 x V: they must be finite
        kv.view(6, -1)[:, (N // 8) * 1024:].zero_()
        nat.check(lib.eqd_embed(g, nat.ptr(emb), nat.ptr(res_l), nat.ptr(res_r), nat.ptr(mu_l), nat.ptr(mu_r),
                                nat.ptr(x_l), nat.ptr(x_r), nat.ptr(h0), nat.ptr(x0), st), 'eqd_embed')
        tc0 = layers[0].dh == nat.H0 and not _LAYER0_FFMA   # 69-wide layer 0 on the tensor cores too
        if tc0:
            x5 = torch.empty(((N + 7) // 8 + 8) * 8, 16, **f32)   # channels 64..68 of K, V, Q; pad rows must be finite
            x5[N:].zero_()
            mu0 = torch.empty(N, nat.H0_PAD, **f32)
            nat.check(lib.eqd_project_tc0(g, C.byref(layers[0].struct), nat.ptr(h0), nat.ptr(pa), nat.ptr(kv), nat.ptr(x5),
                                          st), 'eqd_project_tc0')
        else:
            nat.check(lib.eqd_project(g, C.byref(layers[0].struct), nat.ptr(h0), nat.H0_PAD, nat.ptr(pa), st),
                      'eqd_project')
        h_in, ldh, x_in = h0, nat.H0_PAD, x0
        h_out, x_out = ha, xa
        for li, lay in enumerate(layers):
            nxt = layers[li + 1] if li + 1 < len(layers) else None
            lp = C.byref(lay.struct)
            lpn = C.byref(nxt.struct) if nxt is not None else None
            tmr = stage_timer
            if tmr is not None:
                tmr.begin('edge_stage', li)
            nat.check(lib.eqd_edge_stage(g, lp, nat.ptr(pa), nat.ptr(x_in), nat.ptr(x0), nat.ptr(aggr),
                                         nat.ptr(x_out), nat.ptr(status), st), f'eqd_edge_stage[{li}]')
            if tmr is not None:
                tmr.end('edge_stage', li)
                tmr.begin('node_stage', li)
            if lay.dh == nat.HID:   # tensor-core node stage: attention, node MLP, next layer's projections + K/V blocks
                nat.check(lib.eqd_node_stage_tc(g, lp, lpn, nat.ptr(h_in), nat.ptr(h0), nat.ptr(pa), nat.ptr(aggr),
                                                nat.ptr(kv), nat.ptr(mu), nat.ptr(h_out), nat.ptr(pb), st),
                          f'eqd_node_stage_tc[{li}]')
            elif tc0 and li == 0:   # 69-wide layer 0: 64 tensor-core channels + 5 fp32 ones
                nat.check(lib.eqd_node_stage_tc0(g, lp, lpn, nat.ptr(h0), nat.ptr(pa), nat.ptr(aggr), nat.ptr(kv),
                                                 nat.ptr(x5), nat.ptr(mu0), nat.ptr(h_out), nat.ptr(pb), st),
                          'eqd_node_stage_tc0')
            else:                   # fp32 CUDA-core node stage (fused projections), then K/V blocks
                nat.check(lib.eqd_node_stage(g, lp, lpn, nat.ptr(h_in), ldh, nat.ptr(h0), nat.ptr(pa), nat.ptr(aggr),
                                             nat.ptr(h_out), nat.ptr(pb), st), f'eqd_node_stage[{li}]')
                if nxt is not None:
                    nat.check(lib.eqd_kv_blocks(g, nat.ptr(pb), 320, 192, 256, nat.ptr(kv), st), 'eqd_kv_blocks')
            if tmr is not None:
                tmr.end('node_stage', li)
            pa, pb = pb, pa
            h_in, ldh, x_in = h_out, nat.HID, x_out
            h_out = hb if h_out is ha else ha
            x_out = xb if x_out is xa else xa
        h_fin, x_fin = h_in, x_in
        ws_bytes = lib.eqd_workspace_bytes(N, plan.n_node_tiles, B)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        keyp = torch.empty(2 * B, nat.HEADS, 3, **f64)
        ymean = torch.empty(2 * B, 3, **f64)
        cov = torch.empty(B, 9, **f64)
        nat.check(lib.eqd_keypoints(g, C.byref(head.struct), nat.ptr(h_fin), nat.ptr(x_fin), nat.ptr(ws), ws_bytes,
                                    nat.ptr(keyp), nat.ptr(ymean), nat.ptr(cov), st), 'eqd_keypoints')
        rot, trans = torch.empty(B, 3, 3, **f32), torch.empty(B, 1, 3, **f32)
        lig_out = torch.empty(plan.N_l, 3, **f32)
        sing = torch.empty(B, 3, **f64)
        kab = lambda mask: nat.check(lib.eqd_kabsch_apply(
            g, nat.ptr(cov), nat.ptr(ymean), nat.ptr(x_l), nat.ptr(mask), nat.ptr(rot), nat.ptr(trans),
            nat.ptr(lig_out), nat.ptr(sing), nat.ptr(status), st), 'eqd_kabsch_apply')
        kab(None)
        # status words -> pinned host memory, asynchronously; resolve_status() waits on the event only, so a caller
        # may launch the next forward before looking at this one's flags (bench.py keeps two steps in flight)
        lease = _StatusLease(B + 2)
        status_host = lease.view()
        status_host[:B + 1].copy_(status, non_blocking=True)
        status_host[B + 1:].copy_(plan.unsorted_i32, non_blocking=True)
        status_event = torch.cuda.Event()
        status_event.record()
        out = {'status_lease': lease,'ligand_coors': lig_out, 'keypts': keyp, 'rotation': rot, 'translation': trans, 'h': h_fin,
               'x64': x_fin, 'cov': cov, 'sing': sing, 'status': status, 'unsorted': plan.unsorted, 'kabsch': kab,
               'status_host': status_host, 'status_event': status_event}
        if check_status:
            self.resolve_status(plan, out, kab, log)
        return out

    def resolve_status(self, plan: GraphPlan, out, kab, log=None):
        """The ONE host sync of a forward: reads the status words and replays the reference's
        host-side control flow for flagged pairs (rigid_docking_model.py:570-584)."""
        with torch.cuda.device(self.device):
            try:
                self._resolve_status(plan, out, kab, log)
            finally:
                lease = out.get('status_lease')
                if lease is not None:       # the flags have been read (or the call failed): the buffer may be reused
                    out['status_host'] = out['status_host'].clone()
                    lease.release()

    def _resolve_status(self, plan: GraphPlan, out, kab, log=None):
        out['status_event'].synchronize()
        st_host = out['status_host']
        if int(st_host[-1]) != 0:
            raise UnsortedEdges()
        if int(st_host[plan.n_pairs]) & nat.STATUS_BAD_RESIDUE:
            raise IndexError('res_feat holds a residue index outside [0, 21): index out of range in self '
                             '(nn.Embedding, rigid_docking_model.py:460)')
        if int(st_host[plan.n_pairs]) & nat.STATUS_DEGREE_OVERFLOW:
            raise nat.NativeLibraryError(
                f'a node has more than max_in_degree={plan.struct.max_in_degree} in-edges; '
                'pass the true bound (args["graph_max_neighbor"])')
        pair_st = st_host[:plan.n_pairs]
        if not bool(pair_st.any()):
            return
        if bool((pair_st & nat.STATUS_NAN).any()):
            raise AssertionError('NaN in the Kabsch covariance (rigid_docking_model.py:570)')
        eye_idx = torch.tensor([0, 4, 8], device=self.device)
        for b in torch.nonzero(pair_st & nat.STATUS_SVD_DEGENERATE).reshape(-1).tolist():
            mask = torch.zeros(plan.n_pairs, dtype=torch.int32, device=self.device)
            mask[b] = 1
            num_it = 0
            while True:
                noise = torch.rand(3, 3)  # same CPU-generator draw as the reference (:578)
                out['cov'][b, eye_idx] += torch.diagonal(noise).to(self.device, torch.float64)
                kab(mask)
                num_it += 1
                if num_it > 10:  # the reference gives up before re-testing the 11th attempt (:582-584)
                    if log is not None:
                        log('SVD consistently numerically unstable! Exitting ... ')
                    sys.exit(1)
                if int(out['status'][b].item()) & nat.STATUS_SVD_DEGENERATE == 0:
                    break


class UnsortedEdges(RuntimeError):
    pass
