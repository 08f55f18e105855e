"""CPU: training dropout -- the numpy Philox4x32-10 restatement of the kernels' counter-based masks (tests/dropout_oracle.py)
against the Random123 known-answer vectors, the masked oracles against the unmodified ones (all-ones masks), the
hand-derived backward with masks against torch.autograd, and the host side of the C ABI / binding."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import backward_manual as bm
import dropout_oracle as dm
import golden_io as gio
import iegmn_oracle as orc
import iegmn_oracle_torch as ot
from equidock_public_b200 import _native as nat
from equidock_public_b200 import synthetic


@pytest.mark.parametrize('ctr,key,expect', [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answer_vectors(ctr, key, expect):
    got = dm.philox4x32_10(np.asarray(ctr, np.uint64), np.asarray(key, np.uint64))
    assert tuple(int(v) for v in got) == expect


def test_threshold_and_scale():
    assert dm.threshold(0.25) == 2 ** 30 and dm.threshold(0.0) == 0 and dm.threshold(1.0) == 2 ** 32 - 1
    assert dm.threshold(0.1) == nat.dropout_threshold(0.1)
    assert np.float32(nat.dropout_scale(0.25)) == dm.scale(0.25) == np.float32(4.0 / 3.0)


def test_mask_keep_rate_and_counter_words():
    rows = np.arange(4000)
    k = dm.keep_mask(0x0123456789abcdef, 0.25, 2, 1, rows, 64)
    n = k.size
    assert abs(k.mean() - 0.75) < 5 * np.sqrt(0.25 * 0.75 / n)
    # word j of counter c0 = column 4 c0 + j
    w = dm.philox4x32_10(np.array([3, 17, 4 * 2 + 1, 0], np.uint64), np.asarray(dm.split_key(0x0123456789abcdef), np.uint64))
    assert list(k[17, 12:16]) == [bool(v >= dm.threshold(0.25)) for v in w]


def test_rank_layer_site_and_key_change_the_counter():
    rows = np.arange(256)
    base = dm.keep_mask(77, 0.5, 1, 0, rows, 64)
    for other in (dm.keep_mask(77, 0.5, 1, 0, rows, 64, rank=1), dm.keep_mask(77, 0.5, 2, 0, rows, 64),
                  dm.keep_mask(77, 0.5, 1, 1, rows, 64), dm.keep_mask(78, 0.5, 1, 0, rows, 64)):
        agree = (other == base).mean()
        assert 0.45 < agree < 0.55, agree     # independent streams agree on p^2 + (1-p)^2 = 1/2


def test_every_dropout_symbol_is_declared_and_bound():
    src = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'include', 'eqd_iegmn.h')).read()
    declared = set(re.findall(r'^\s*(?:int|size_t|void\*?|float)\s+(eqd_\w+)\s*\(', src, flags=re.M))
    new = {'eqd_iegmn_forward_dropout', 'eqd_dropout_mask', 'eqd_bwd_edge_dropout', 'eqd_bwd_node_mlp_dropout',
           'eqd_bwd_head_dropout'}
    assert new <= declared and new <= set(nat.PROTOTYPES)
    assert re.search(r'#define EQD_ABI_VERSION %d\b' % nat.ABI_VERSION, src)
    body = re.search(r'typedef struct eqd_dropout \{(.*?)\} eqd_dropout;', src, flags=re.S).group(1)
    fields = re.findall(r'(\w+);', body)
    assert fields == [f[0] for f in nat.EqdDropout._fields_]
    assert C.sizeof(nat.EqdDropout) == 24


def test_binding_dropout_state_on_cpu():
    d = nat.Dropout(0.25, 'cpu', rank=3, key=torch.tensor([0x0123456789abcdef], dtype=torch.int64))
    assert d.struct.threshold == 2 ** 30 and d.struct.rank == 3 and d.struct.key == d.key.data_ptr()
    with pytest.raises(ValueError):
        nat.Dropout(1.0, 'cpu')
    g0 = torch.get_rng_state()
    nat.Dropout(0.5, 'cpu')        # a CPU key draws from the CPU generator; on a GPU the CUDA generator is used
    assert not torch.equal(g0, torch.get_rng_state())


def test_model_reads_p_from_the_dropout_modules():
    args = dict(gio.load_args('dips'))
    args['dropout'] = 0.25
    model = gio.build_model('dips', 'cpu', args=args).train()
    iegmn = model.iegmn_original
    assert iegmn.dropout_p() == 0.25
    model.eval()
    assert iegmn.dropout_p() == 0.0
    model.train()
    iegmn.iegmn_layers[1].node_mlp[1].p = 0.1
    with pytest.raises(NotImplementedError):
        iegmn.dropout_p()
    for m in model.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 1.0
    with pytest.raises(NotImplementedError):
        iegmn.dropout_p()
    with pytest.raises(NotImplementedError):   # the per-layer operator keeps raising in train mode with p > 0
        iegmn.iegmn_layers[0]._check_mode()


@pytest.mark.parametrize('ds', ['db5', 'dips'])
def test_oracles_with_all_ones_masks_equal_no_masks(ds):
    names, pairs, outs, _ = gio.load_pairs(ds)
    lig, rec = pairs[names[0]]
    sd, args = gio.load_checkpoint(ds), gio.load_args(ds)
    cfg = orc.OracleConfig.from_args(args)
    sizes = [(len(lig['x']), len(rec['x']), len(lig['src']), len(rec['src']))]
    ones = {k: np.ones_like(v) for k, v in dm.pair_masks(5, 0.25, cfg.n_layers, sizes)[0].items()}
    f = lambda o: (1e-3 * o['ligand_coors'], 1e-3 * o['keypts_ligand'], 1e-3 * o['keypts_receptor'])
    shared = bool(args['shared_layers'])
    ga, oa = bm.full_backward(sd, cfg, lig, rec, f, shared)
    for masks in (None, ones):
        gb, ob = dm.full_backward(sd, cfg, lig, rec, f, shared, masks=masks)
        assert all(np.array_equal(oa[k], ob[k]) for k in oa)
        assert all(np.array_equal(ga[k], gb[k]) for k in ga)
    ref = orc.forward_pair(sd, cfg, lig, rec)
    assert np.abs(ref['ligand_coors'] - ob['ligand_coors']).max() < 1e-8
    model = ot.TorchOracle(sd, cfg.n_layers, cfg.skip_weight_h, cfg.x_connection_init, cfg.slope, cfg.num_att_heads,
                           dtype=torch.float64)
    masked = dm.TorchOracle(sd, cfg.n_layers, cfg.skip_weight_h, cfg.x_connection_init, cfg.slope, cfg.num_att_heads,
                            dtype=torch.float64)
    ta = model.forward_pair(lig, rec)
    with torch.no_grad():
        for masks in (None, ones):
            tb = masked.forward_pair_grad(lig, rec, masks=masks)
            assert all(torch.equal(ta[k], tb[k]) for k in ta)


@pytest.mark.parametrize('ds', ['db5', 'dips'])
def test_manual_backward_with_dropout_equals_autograd_ragged_batch(ds):
    """Random masks (p = 0.25) of a ragged batch of 3 (tile boundaries 128 + 1, 128 + 3), sliced per pair: the hand-derived
    backward equals torch.autograd on the torch restatement with the same multipliers."""
    sd, args = gio.load_checkpoint(ds), gio.load_args(ds)
    cfg = orc.OracleConfig.from_args(args)
    rng = np.random.default_rng(11)
    pairs = [synthetic.synthetic_pair(rng, a, b, 10) for a, b in [(40, 131), (129, 20), (64, 64)]]
    sizes = [(len(l['x']), len(r['x']), len(l['src']), len(r['src'])) for l, r in pairs]
    masks = dm.pair_masks(0x243f6a8885a308d3, 0.25, cfg.n_layers, sizes)
    model = dm.TorchOracle(sd, cfg.n_layers, cfg.skip_weight_h, cfg.x_connection_init, cfg.slope, cfg.num_att_heads,
                           dtype=torch.float64)
    psd = model.parameters_for_grad()
    shared = bool(args['shared_layers'])
    total = None
    for (lig, rec), m in zip(pairs, masks):
        tgt = {'c': rng.normal(0, 5, (len(lig['x']), 3)), 'yl': rng.normal(0, 10, (50, 3)), 'yr': rng.normal(0, 10, (50, 3))}
        f = lambda o, t=tgt: (2e-3 * (o['ligand_coors'] - t['c']), 2e-3 * (o['keypts_ligand'] - t['yl']),
                              2e-3 * (o['keypts_receptor'] - t['yr']))
        g, out = dm.full_backward(sd, cfg, lig, rec, f, shared, masks=m)
        total = g if total is None else {k: total[k] + g[k] for k in g}
        o = model.forward_pair_grad(lig, rec, masks=m)
        assert np.abs(out['ligand_coors'] - o['ligand_coors'].detach().numpy()).max() < 1e-8
        t = lambda a: torch.as_tensor(a, dtype=torch.float64)
        (1e-3 * ((o['ligand_coors'] - t(tgt['c'])) ** 2).sum() + 1e-3 * ((o['keypts_ligand'] - t(tgt['yl'])) ** 2).sum()
         + 1e-3 * ((o['keypts_receptor'] - t(tgt['yr'])) ** 2).sum()).backward()
    for name, leaf in psd.items():
        if not leaf.is_floating_point():
            continue
        ref = leaf.grad.numpy() if leaf.grad is not None else np.zeros(tuple(leaf.shape))
        if shared and '.iegmn_layers.' in name and int(name.split('.iegmn_layers.')[1].split('.')[0]) >= 1:
            suffix = name.split('.iegmn_layers.')[1].split('.', 1)[1]
            ref = sum(psd[f'iegmn_original.iegmn_layers.{j}.{suffix}'].grad.numpy() for j in range(1, cfg.n_layers))
        got = total[name].reshape(ref.shape)
        scale = max(np.abs(ref).max(), 1e-12)
        assert np.abs(got - ref).max() <= 1e-7 * scale + 1e-12, (name, np.abs(got - ref).max(), scale)
    # the masks are not trivial: dropout changes the gradients
    lig, rec = pairs[0]
    f0 = lambda o: (1e-3 * o['ligand_coors'], 1e-3 * o['keypts_ligand'], 1e-3 * o['keypts_receptor'])
    g0, _ = bm.full_backward(sd, cfg, lig, rec, f0, shared)
    g1, _ = dm.full_backward(sd, cfg, lig, rec, f0, shared, masks=masks[0])
    assert not np.allclose(g0['iegmn_original.mlp_h_mean_ROT.0.weight'], g1['iegmn_original.mlp_h_mean_ROT.0.weight'])
