"""TEST INFRASTRUCTURE -- fp64 oracles of TRAINING WITH DROPOUT, next to the unmodified ones in ``oracle/``.

1. The engine's counter-based dropout masks (csrc/dropout.cuh) restated in numpy, bit for bit: Philox4x32-10 (Salmon et
   al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123 constants), vectorised over rows.  Element
   (row, col) of site `site` in layer `layer` (site 3, mlp_h_mean_ROT, uses layer = n_layers):

       counter = {col // 4, row, 4 * layer + site, rank},  key = {key64 & 0xffffffff, key64 >> 32}
       word    = output word (col % 4) of Philox4x32-10(counter, key)
       keep    = word >= threshold(p),   threshold(p) = min(round(p * 2^32), 2^32 - 1)
       multiplier = fp32(1 / (1 - p)) if keep else 0

   Rows are global edge ids in the plan's CSR order (sites 0: edge_mlp, 1: coors_mlp) or global node ids (2: node_mlp,
   3: mlp_h_mean_ROT).

2. The forward + hand-derived backward of ``oracle/backward_manual.py`` and the torch restatement of
   ``oracle/iegmn_oracle_torch.py`` with optional per-site dropout multipliers: ``masks`` = {(layer, site, side): array
   rows x width of m * s} (side 0 ligand, 1 receptor; a missing key = no dropout there).  Each mask multiplies the
   LeakyReLU output of its site, which equals the reference's dropout-then-LeakyReLU (LeakyReLU is positively
   homogeneous): a1 = m0 lrelu(z1), c3 = m1 lrelu(z3), a5 = m2 lrelu(u5), qbar = mean(m3 lrelu(W_m h + b_m)); the backward
   multiplies the same m into dz1, dz3, du and dpre.  Only the functions the masks touch are restated here; everything
   else is the unmodified oracle code.  With all-ones masks the results equal the unmodified oracles exactly
   (tests/test_dropout_host.py).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

import backward_manual as bm
import iegmn_oracle_torch as ot
from backward_manual import ln_backward, ln_forward, lrelu_grad, seg_mean
from iegmn_oracle import SIGMAS, LayerParams, leaky_relu, linear

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: uint32-compatible array (..., 4); key: (..., 2) (broadcast).  Returns uint32 (..., 4)."""
    c = [np.asarray(ctr, dtype=np.uint64)[..., i] & _MASK32 for i in range(4)]
    key = np.asarray(key, dtype=np.uint64)
    k0, k1 = key[..., 0] & _MASK32, key[..., 1] & _MASK32
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(W0)) & _MASK32
            k1 = (k1 + np.uint64(W1)) & _MASK32
        p0 = np.uint64(M0) * c[0]
        p1 = np.uint64(M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, axis=-1).astype(np.uint32)


def threshold(p: float) -> int:
    return min(int(round(float(p) * 2.0 ** 32)), 2 ** 32 - 1)


def scale(p: float) -> np.float32:
    return np.float32(1.0 / (1.0 - float(p)))


def split_key(key64: int):
    key64 = int(key64) & (2 ** 64 - 1)
    return key64 & 0xFFFFFFFF, key64 >> 32


def keep_mask(key64: int, p: float, layer: int, site: int, rows, cols: int, rank: int = 0) -> np.ndarray:
    """bool [len(rows)][cols]: keep bits of the given global rows (any int array), columns 0..cols-1."""
    rows = np.asarray(rows, dtype=np.int64).reshape(-1)
    nc4 = (cols + 3) // 4
    ctr = np.zeros((rows.shape[0], nc4, 4), dtype=np.uint64)
    ctr[..., 0] = np.arange(nc4, dtype=np.uint64)[None, :]
    ctr[..., 1] = rows.astype(np.uint64)[:, None]
    ctr[..., 2] = 4 * int(layer) + int(site)
    ctr[..., 3] = int(rank)
    words = philox4x32_10(ctr, np.asarray(split_key(key64), dtype=np.uint64))
    return words.reshape(rows.shape[0], nc4 * 4)[:, :cols] >= np.uint32(threshold(p))


def multiplier(key64: int, p: float, layer: int, site: int, rows, cols: int, rank: int = 0) -> np.ndarray:
    """float64 [len(rows)][cols]: the dropout multiplier m * s (fp32 scale, widened) of every element."""
    return keep_mask(key64, p, layer, site, rows, cols, rank).astype(np.float64) * float(scale(p))


def pair_masks(key64: int, p: float, n_layers: int, sizes, rank: int = 0, dh0: int = 69):
    """Per-pair dropout multipliers of a batch, for the per-pair oracles (iegmn_oracle.drop_mult layout): one dict per pair,
    keyed (layer, site, side).  ``sizes`` = [(N_l, N_r, E_l, E_r)] of the pairs in batch order; the batch numbers ligand
    nodes / edges of all pairs first, then the receptor ones (include/eqd_iegmn.h), and the per-pair masks are slices of
    the batch masks.  Site 2 of layer 0 is ``dh0`` wide (the 69-wide first layer), every other site 64."""
    sizes = [tuple(int(v) for v in s) for s in sizes]
    n_l, n_r, e_l, e_r = (np.asarray([s[i] for s in sizes], dtype=np.int64) for i in range(4))
    node0 = [np.concatenate([[0], np.cumsum(n_l)[:-1]]), n_l.sum() + np.concatenate([[0], np.cumsum(n_r)[:-1]])]
    edge0 = [np.concatenate([[0], np.cumsum(e_l)[:-1]]), e_l.sum() + np.concatenate([[0], np.cumsum(e_r)[:-1]])]
    out = []
    for b in range(len(sizes)):
        m = {}
        for side, (nn, ne) in enumerate(((n_l[b], e_l[b]), (n_r[b], e_r[b]))):
            erows = edge0[side][b] + np.arange(ne)
            nrows = node0[side][b] + np.arange(nn)
            for li in range(n_layers):
                m[(li, 0, side)] = multiplier(key64, p, li, 0, erows, 64, rank)
                m[(li, 1, side)] = multiplier(key64, p, li, 1, erows, 64, rank)
                m[(li, 2, side)] = multiplier(key64, p, li, 2, nrows, dh0 if li == 0 else 64, rank)
            m[(n_layers, 3, side)] = multiplier(key64, p, n_layers, 3, nrows, 64, rank)
        out.append(m)
    return out


# ---- the oracles with dropout multipliers -----------------------------------------------------------------------------

def drop_mult(masks, layer, site, side):
    """Multiplier array (m * s) of (layer, site, side), or 1.0 (no dropout)."""
    if masks is None:
        return 1.0
    m = masks.get((layer, site, side))
    return 1.0 if m is None else m


def layer_forward(p: LayerParams, cfg, sides, masks=None, layer=0):
    """backward_manual.layer_forward with the site 0 / 1 / 2 multipliers (kept in the caches as m0, m1, m2)."""
    slope, dh = cfg.slope, p.h_dim
    caches = []
    for s in sides:
        h = s['h']
        c = {'h': h, 'x': s['x'], 'h0': s['h0'], 'he': s['he'], 'src': s['src'], 'dst': s['dst'], 'x_orig': s['x_orig']}
        c['qpre'], c['kpre'] = linear(h, p.wq), linear(h, p.wk)
        c['q'], c['k'], c['v'] = leaky_relu(c['qpre'], slope), leaky_relu(c['kpre'], slope), linear(h, p.wv)
        c['psrc'] = linear(h, p.edge_w1[:, 0:dh])
        c['pdst'] = linear(h, p.edge_w1[:, dh:2 * dh], p.edge_b1)
        caches.append(c)
    for i, c in enumerate(caches):
        o = caches[1 - i]
        src, dst, n = c['src'], c['dst'], c['x'].shape[0]
        c['m0'], c['m1'], c['m2'] = (drop_mult(masks, layer, site, i) for site in range(3))
        c['xrel'] = c['x'][src] - c['x'][dst]
        d2 = (c['xrel'] ** 2).sum(1, keepdims=True)
        c['rbf'] = np.concatenate([np.exp(-d2 / sg) for sg in SIGMAS], 1)
        c['ein'] = np.concatenate([c['he'], c['rbf']], 1)
        c['z1'] = c['psrc'][src] + c['pdst'][dst] + c['ein'] @ p.edge_w1[:, 2 * dh:].T
        c['n1'], c['nhat1'], c['rstd1'] = ln_forward(leaky_relu(c['z1'], slope) * c['m0'], p.edge_ln_g, p.edge_ln_b)
        c['msg'] = linear(c['n1'], p.edge_w2, p.edge_b2)
        c['z3'] = linear(c['msg'], p.coor_w1, p.coor_b1)
        c['c3'] = leaky_relu(c['z3'], slope) * c['m1']
        c['phi'] = linear(c['c3'], p.coor_w2, p.coor_b2)
        c['aggr'], c['deg'] = seg_mean(c['msg'], dst, n)
        xupd, _ = seg_mean(c['xrel'] * c['phi'], dst, n)
        c['x_new'] = cfg.x_connection_init * c['x_orig'] + (1 - cfg.x_connection_init) * c['x'] + xupd
        S = c['q'] @ o['k'].T
        S = S - S.max(1, keepdims=True)
        P = np.exp(S)
        c['P'] = P / P.sum(1, keepdims=True)
        c['mu'] = c['P'] @ o['v']
        c['inp'] = np.concatenate([c['h'], c['aggr'], c['mu'], c['h0']], 1)
        c['u5'] = linear(c['inp'], p.node_w1, p.node_b1)
        c['n5'], c['nhat5'], c['rstd5'] = ln_forward(leaky_relu(c['u5'], slope) * c['m2'], p.node_ln_g, p.node_ln_b)
        o6 = linear(c['n5'], p.node_w2, p.node_b2)
        c['skip'] = p.h_dim == p.out_dim
        c['h_new'] = cfg.skip_weight_h * o6 + (1 - cfg.skip_weight_h) * c['h'] if c['skip'] else o6
    return caches


def node_mlp_bwd(p, cfg, c, dh_new, G):
    """backward_manual.node_mlp_bwd with du = m2 lrelu'(u5) da."""
    dh_ = p.h_dim
    do = cfg.skip_weight_h * dh_new if c['skip'] else dh_new
    dh = (1 - cfg.skip_weight_h) * dh_new if c['skip'] else np.zeros_like(c['h'])
    G['node_w2'] += do.T @ c['n5']
    G['node_b2'] += do.sum(0)
    da, dg, db = ln_backward(do @ p.node_w2, c['nhat5'], c['rstd5'], p.node_ln_g)
    G['node_ln_g'] += dg
    G['node_ln_b'] += db
    du = da * lrelu_grad(c['u5'], cfg.slope) * c['m2']
    G['node_w1'] += du.T @ c['inp']
    G['node_b1'] += du.sum(0)
    dinp = du @ p.node_w1
    return dh + dinp[:, 0:dh_], dinp[:, dh_:dh_ + 64], dinp[:, dh_ + 64:2 * dh_ + 64], dinp[:, 2 * dh_ + 64:]


def edge_bwd(p, cfg, c, daggr, dx_new, G):
    """backward_manual.edge_bwd with dz3 = m1 lrelu'(z3) dphi w4 and dz1 = m0 lrelu'(z1) da."""
    slope, dh_ = cfg.slope, p.h_dim
    dst = c['dst']
    deg = np.maximum(c['deg'], 1)[dst][:, None]
    dmsg = daggr[dst] / deg
    dxm = dx_new[dst] / deg
    dphi = (c['xrel'] * dxm).sum(1, keepdims=True)
    dxrel = c['phi'] * dxm
    G['coor_w2'] += dphi.T @ c['c3']
    G['coor_b2'] += dphi.sum(0)
    dz3 = (dphi @ p.coor_w2) * lrelu_grad(c['z3'], slope) * c['m1']
    G['coor_w1'] += dz3.T @ c['msg']
    G['coor_b1'] += dz3.sum(0)
    dmsg = dmsg + dz3 @ p.coor_w1
    G['edge_w2'] += dmsg.T @ c['n1']
    G['edge_b2'] += dmsg.sum(0)
    da, dg, db = ln_backward(dmsg @ p.edge_w2, c['nhat1'], c['rstd1'], p.edge_ln_g)
    G['edge_ln_g'] += dg
    G['edge_ln_b'] += db
    dz1 = da * lrelu_grad(c['z1'], slope) * c['m0']
    G['edge_w1'][:, 2 * dh_:] += dz1.T @ c['ein']
    drbf = dz1 @ p.edge_w1[:, 2 * dh_ + 27:]
    dd2 = (drbf * c['rbf'] * (-1.0 / np.asarray(SIGMAS))).sum(1, keepdims=True)
    return dz1, dxrel + 2.0 * c['xrel'] * dd2


def layer_backward(p, cfg, caches, dh_new, dx_new, G, stages=None):
    """backward_manual.layer_backward over the masked node / edge stages (attention, gather, projections unchanged)."""
    nm = [node_mlp_bwd(p, cfg, c, dh_new[i], G) for i, c in enumerate(caches)]
    att = bm.attn_bwd(cfg, caches, [m[2] for m in nm])
    out = []
    for i, c in enumerate(caches):
        dh_part, daggr, dmu, dh0 = nm[i]
        dz1, dxrel = edge_bwd(p, cfg, c, daggr, dx_new[i], G)
        dpsrc, dpdst, dx = bm.edge_gather(cfg, c, dz1, dxrel, dx_new[i])
        dqpre, dkpre, dv = att[i]
        dh = dh_part + bm.proj_bwd(p, c, dpsrc, dpdst, dqpre, dkpre, dv, G)
        out.append((dh, dx, dh0))
        if stages is not None:
            stages.append({'side': i, 'dh_part': dh_part, 'daggr': daggr, 'dmu': dmu, 'dh0': dh0, 'dz1': dz1, 'dxrel': dxrel,
                           'dpsrc': dpsrc, 'dpdst': dpdst, 'dx': dx, 'dqpre': dqpre, 'dkpre': dkpre, 'dv': dv, 'dh': dh})
    return out


def head_forward(sd, cfg, h_l, x_l, h_r, x_r, masks=None):
    """backward_manual.head_forward with qbar = mean(m3 lrelu(W_m h + b_m)) (m3 kept as c['m3'])."""
    c = bm.head_forward(sd, cfg, h_l, x_l, h_r, x_r)
    c['m3'] = [drop_mult(masks, cfg.n_layers, 3, i) for i in range(2)]
    if masks is None:
        return c
    H, X = c['H'], c['X']
    c['qbar'] = [(leaky_relu(pr, cfg.slope) * m).mean(0) for pr, m in zip(c['pre'], c['m3'])]
    for i in range(2):                    # everything downstream of qbar, as in backward_manual.head_forward
        qb = c['qbar'][1 - i]
        c['r'][i] = np.einsum('ked,d->ke', c['wq'], qb)
        c['u'][i] = np.einsum('ked,ke->kd', c['wk'], c['r'][i]) / math.sqrt(64)
        lg = c['u'][i] @ H[i].T
        lg = lg - lg.max(1, keepdims=True)
        e = np.exp(lg)
        c['att'][i] = e / e.sum(1, keepdims=True)
        c['Y'][i] = c['att'][i] @ X[i]
    y_l, y_r = c['Y']
    c['ym'] = [y_l.mean(0), y_r.mean(0)]
    A = (y_r - c['ym'][1]).T @ (y_l - c['ym'][0])
    U, S, Vt = np.linalg.svd(A)
    D = np.diag([1., 1., np.sign(np.linalg.det(A))])
    c.update(A=A, U=U, S=S, Vt=Vt, D=D)
    c['T'] = U @ D @ Vt
    c['b'] = c['ym'][1] - c['T'] @ c['ym'][0]
    return c


def keypoints_bwd(cfg, c, dY, G):
    """backward_manual.keypoints_bwd with dpre = m3 lrelu'(pre) dqbar / n."""
    H, X = c['H'], c['X']
    dh = [np.zeros_like(H[0]), np.zeros_like(H[1])]
    dx = [None, None]
    dqbar = [np.zeros(64), np.zeros(64)]
    for i in range(2):
        att, Y = c['att'][i], c['Y'][i]
        dx[i] = att.T @ dY[i]
        dlog = att * (dY[i] @ X[i].T - (dY[i] * Y).sum(1, keepdims=True))
        dh[i] += dlog.T @ c['u'][i]
        du = dlog @ H[i]
        a = np.einsum('ked,kd->ke', c['wk'], du) / math.sqrt(64)
        G['wk'] += np.einsum('ke,kd->ked', c['r'][i], du) / math.sqrt(64)
        G['wq'] += np.einsum('ke,d->ked', a, c['qbar'][1 - i])
        dqbar[1 - i] += np.einsum('ked,ke->d', c['wq'], a)
    for i in range(2):
        n = H[i].shape[0]
        dpre = (dqbar[i] / n)[None, :] * np.where(c['pre'][i] > 0, 1.0, cfg.slope) * c['m3'][i]
        G['wm'] += dpre.T @ H[i]
        G['bm'] += dpre.sum(0)
        dh[i] += dpre @ c['wm']
    return dh, dx


def full_backward(sd, cfg, ligand, receptor, loss_grads, shared_layers: bool, stages=None, masks=None):
    """backward_manual.full_backward (forward + manual backward of ONE pair) with dropout multipliers ``masks``."""
    f = lambda a: np.asarray(a, np.float64)
    emb = f(sd['iegmn_original.residue_emb_layer.weight'])
    sides, idxs = [], []
    for s, ck in ((ligand, 'new_x'), (receptor, 'x')):
        idx = np.asarray(s['res_feat']).reshape(-1).astype(np.int64)
        idxs.append(idx)
        h0 = np.concatenate([emb[idx], np.log(f(s['mu_r_norm']))], 1)
        x0 = f(s[ck])
        sides.append({'x': x0, 'x_orig': x0, 'h': h0, 'h0': h0, 'he': f(s['he']),
                      'src': np.asarray(s['src']).astype(np.int64), 'dst': np.asarray(s['dst']).astype(np.int64)})
    params, all_caches = [], []
    for li in range(cfg.n_layers):
        p = LayerParams(sd, f'iegmn_original.iegmn_layers.{li}.', np.float64)
        caches = layer_forward(p, cfg, sides, masks, li)
        for s, c in zip(sides, caches):
            s['x'], s['h'] = c['x_new'], c['h_new']
        params.append(p)
        all_caches.append(caches)
    hc = head_forward(sd, cfg, sides[0]['h'], sides[0]['x'], sides[1]['h'], sides[1]['x'], masks)
    x_in = sides[0]['x_orig']
    out = {'ligand_coors': (hc['T'] @ x_in.T).T + hc['b'], 'keypts_ligand': hc['Y'][0], 'keypts_receptor': hc['Y'][1],
           'rotation': hc['T'], 'translation': hc['b'].reshape(1, 3)}
    dcoors, dYl, dYr = loss_grads(out)
    GH = {'wm': np.zeros((64, 64)), 'bm': np.zeros(64), 'wk': np.zeros_like(hc['wk']), 'wq': np.zeros_like(hc['wq'])}
    dY = bm.kabsch_bwd(hc, x_in, dcoors, (dYl, dYr))
    dh, dx = keypoints_bwd(cfg, hc, dY, GH)
    if stages is not None:
        stages.append({'head': True, 'dY': dY, 'dh': dh, 'dx': dx})
    grads = {'iegmn_original.mlp_h_mean_ROT.0.weight': GH['wm'], 'iegmn_original.mlp_h_mean_ROT.0.bias': GH['bm'],
             'iegmn_original.att_mlp_key_ROT.0.weight': GH['wk'].reshape(-1, 64),
             'iegmn_original.att_mlp_query_ROT.0.weight': GH['wq'].reshape(-1, 64)}
    dh0 = [np.zeros_like(s['h0']) for s in sides]
    names = {'edge_w1': 'edge_mlp.0.weight', 'edge_b1': 'edge_mlp.0.bias', 'edge_ln_g': 'edge_mlp.3.weight',
             'edge_ln_b': 'edge_mlp.3.bias', 'edge_w2': 'edge_mlp.4.weight', 'edge_b2': 'edge_mlp.4.bias',
             'wq': 'att_mlp_Q.0.weight', 'wk': 'att_mlp_K.0.weight', 'wv': 'att_mlp_V.0.weight',
             'node_w1': 'node_mlp.0.weight', 'node_b1': 'node_mlp.0.bias', 'node_ln_g': 'node_mlp.3.weight',
             'node_ln_b': 'node_mlp.3.bias', 'node_w2': 'node_mlp.4.weight', 'node_b2': 'node_mlp.4.bias',
             'coor_w1': 'coors_mlp.0.weight', 'coor_b1': 'coors_mlp.0.bias', 'coor_w2': 'coors_mlp.4.weight',
             'coor_b2': 'coors_mlp.4.bias'}
    layer_G = {}
    for li in reversed(range(cfg.n_layers)):
        key = 1 if (shared_layers and li >= 1) else li
        G = layer_G.setdefault(key, bm.zero_layer_grads(params[li]))
        st = [] if stages is not None else None
        res = layer_backward(params[li], cfg, all_caches[li], dh, dx, G, st)
        dh, dx = [r[0] for r in res], [r[1] for r in res]
        for i in range(2):
            dh0[i] += res[i][2]
        if stages is not None:
            stages.append({'layer': li, 'sides': st})
    for i in range(2):
        dh0[i] += dh[i]
    demb = np.zeros_like(emb)
    for i in range(2):
        np.add.at(demb, idxs[i], dh0[i][:, :64])
    grads['iegmn_original.residue_emb_layer.weight'] = demb
    for li in range(cfg.n_layers):
        key = 1 if (shared_layers and li >= 1) else li
        for short, nm in names.items():
            grads[f'iegmn_original.iegmn_layers.{li}.{nm}'] = layer_G[key][short]
    return grads, out


class TorchOracle(ot.TorchOracle):
    """iegmn_oracle_torch.TorchOracle (the autograd reference of the backward) with dropout multipliers."""

    def _drop(self, masks, layer, site, side):
        m = None if masks is None else masks.get((layer, site, side))
        return 1.0 if m is None else torch.as_tensor(m).to(self.dtype)

    def _layer(self, li, sides, masks=None):
        p = lambda k: self.sd[f'iegmn_original.iegmn_layers.{li}.{k}']
        lr = lambda t: F.leaky_relu(t, self.slope)
        q = [lr(F.linear(s['h'], p('att_mlp_Q.0.weight'))) for s in sides]
        k = [lr(F.linear(s['h'], p('att_mlp_K.0.weight'))) for s in sides]
        v = [F.linear(s['h'], p('att_mlp_V.0.weight')) for s in sides]
        new = []
        for i, s in enumerate(sides):
            o = 1 - i
            x, h, src, dst = s['x'], s['h'], s['src'], s['dst']
            n = x.shape[0]
            x_rel = x[src] - x[dst]
            d2 = (x_rel ** 2).sum(1, keepdim=True)
            rbf = torch.cat([torch.exp(-d2 / sg) for sg in SIGMAS], dim=-1)
            cat = torch.cat([h[src], h[dst], s['he'], rbf], dim=-1)
            a = lr(F.linear(cat, p('edge_mlp.0.weight'), p('edge_mlp.0.bias'))) * self._drop(masks, li, 0, i)
            a = F.layer_norm(a, (a.shape[1],), p('edge_mlp.3.weight'), p('edge_mlp.3.bias'))
            msg = F.linear(a, p('edge_mlp.4.weight'), p('edge_mlp.4.bias'))
            mu = torch.softmax(q[i] @ k[o].t(), dim=1) @ v[o]
            c = lr(F.linear(msg, p('coors_mlp.0.weight'), p('coors_mlp.0.bias'))) * self._drop(masks, li, 1, i)
            coef = F.linear(c, p('coors_mlp.4.weight'), p('coors_mlp.4.bias'))
            x_new = self.eta * s['x0'] + (1. - self.eta) * x + ot._segment_mean(x_rel * coef, dst, n)
            inp = torch.cat([h, ot._segment_mean(msg, dst, n), mu, s['h0']], dim=-1)
            hid = lr(F.linear(inp, p('node_mlp.0.weight'), p('node_mlp.0.bias'))) * self._drop(masks, li, 2, i)
            hid = F.layer_norm(hid, (hid.shape[1],), p('node_mlp.3.weight'), p('node_mlp.3.bias'))
            h_new = F.linear(hid, p('node_mlp.4.weight'), p('node_mlp.4.bias'))
            if h_new.shape[1] == h.shape[1]:
                h_new = self.sk * h_new + (1. - self.sk) * h
            new.append((x_new, h_new))
        for s, (x_new, h_new) in zip(sides, new):
            s['x'], s['h'] = x_new, h_new

    def forward_pair_grad(self, lig, rec, masks=None):
        sd, dt = self.sd, self.dtype
        emb = sd['iegmn_original.residue_emb_layer.weight']
        sides = []
        for s, ck in ((lig, 'new_x'), (rec, 'x')):
            idx = torch.as_tensor(s['res_feat']).reshape(-1).long()
            h0 = torch.cat([emb[idx], torch.log(torch.as_tensor(s['mu_r_norm']).to(dt))], dim=1)
            x0 = torch.as_tensor(s[ck]).to(dt)
            sides.append({'x': x0, 'x0': x0, 'h': h0, 'h0': h0, 'he': torch.as_tensor(s['he']).to(dt),
                          'src': torch.as_tensor(s['src']).long(), 'dst': torch.as_tensor(s['dst']).long()})
        for li in range(self.L):
            self._layer(li, sides, masks)
        l, r = sides
        g = lambda k: sd['iegmn_original.' + k]
        d = l['h'].shape[1]
        mean = lambda h, m: (F.leaky_relu(F.linear(h, g('mlp_h_mean_ROT.0.weight'), g('mlp_h_mean_ROT.0.bias')),
                                          self.slope) * m).mean(0, keepdim=True)
        m_l, m_r = mean(l['h'], self._drop(masks, self.L, 3, 0)), mean(r['h'], self._drop(masks, self.L, 3, 1))

        def keypts(hk, mq, z):
            keys = F.linear(hk, g('att_mlp_key_ROT.0.weight')).view(-1, self.K, d).transpose(0, 1)
            qry = F.linear(mq, g('att_mlp_query_ROT.0.weight')).view(1, self.K, d).transpose(0, 1).transpose(1, 2)
            att = torch.softmax(keys @ qry / math.sqrt(d), dim=1).view(self.K, -1)
            return att @ z

        y_r, y_l = keypts(r['h'], m_l, r['x']), keypts(l['h'], m_r, l['x'])
        yr_m, yl_m = y_r.mean(0, keepdim=True), y_l.mean(0, keepdim=True)
        A = (y_r - yr_m).t() @ (y_l - yl_m)
        U, S, Vt = torch.linalg.svd(A)
        corr = torch.diag(torch.tensor([1., 1., float(torch.sign(torch.det(A.detach())))], dtype=dt))
        T = (U @ corr) @ Vt
        b = yr_m - (T @ yl_m.t()).t()
        return {'ligand_coors': (T @ l['x0'].t()).t() + b, 'rotation': T, 'translation': b,
                'keypts_ligand': y_l, 'keypts_receptor': y_r}
