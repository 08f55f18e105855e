"""CPU: the on-disk formats (SURVEY 8f rank 4): flat pair archive round trip incl. labels, PDB writer round trip,
checkpoint dict compatible with the reference's loader."""
import numpy as np
import torch

import golden_io as gio
from equidock_public_b200 import formats


def test_pair_archive_round_trip(tmp_path):
    names, pairs, _, _ = gio.load_pairs('dips')
    pl = [pairs[n] for n in names]
    rng = np.random.default_rng(0)
    labels = [{'pocket_coors': rng.normal(size=(5 + 3 * i, 3)), 'bound_lig': p[0]['x'], 'bound_rec': p[1]['x']} for i, p in enumerate(pl)]
    path = str(tmp_path / 'dips.eqd')
    formats.save_pairs(path, pl, labels, meta={'dataset': 'dips'})
    arc = formats.PairArchive(path)
    assert len(arc) == len(pl) and arc.a.meta['dataset'] == 'dips'
    for i, (lig, rec) in enumerate(pl):
        a, b = arc.pair(i)
        for got, ref in ((a, lig), (b, rec)):
            for k in ('src', 'dst', 'he', 'x', 'mu_r_norm'):
                assert np.array_equal(got[k], ref[k]), k
            assert np.array_equal(got['res_feat'], ref['res_feat'])
        assert np.array_equal(a['new_x'], lig['new_x'])
        lab = arc.labels(i)
        assert np.allclose(lab['pocket_coors'], labels[i]['pocket_coors'].astype(np.float32)) and lab['bound_lig'].shape == lig['x'].shape
    g = arc.batch([2, 0])
    assert g.batch_size == 2 and g.num_nodes('ligand') == pl[2][0]['x'].shape[0] + pl[0][0]['x'].shape[0]
    ref = gio.make_batch([pl[2], pl[0]])
    assert torch.equal(g.edges['ll'].data['he'], ref.edges['ll'].data['he'])
    assert torch.equal(g.edges(etype='rr')[0], ref.edges(etype='rr')[0])


def test_pdb_writer_round_trip_and_columns(tmp_path):
    src = tmp_path / 'in.pdb'
    src.write_text('HEADER    TEST\n'
                   'ATOM      1  N   MET A   1      27.340  24.430   2.614  1.00  9.67           N  \n'
                   'ATOM      2  CA  MET A   1      26.266  25.413   2.842  1.00 10.38           C  \n'
                   'HETATM    3  O   HOH A 101      -1.000  -2.000  -3.000  1.00  0.00           O  \n'
                   'ATOM      3  C   MET A   1      26.913  26.639   3.531  1.00  9.62           C  \n'
                   'END\n')
    R = np.array([[0., -1, 0], [1, 0, 0], [0, 0, 1]])
    formats.apply_rigid_to_pdb(str(src), str(tmp_path / 'out.pdb'), R, [1.0, 2.0, -300.5])
    lines, xyz = formats.read_pdb_atoms(str(tmp_path / 'out.pdb'))
    assert len(lines) == 3 and lines[0][:30] == 'ATOM      1  N   MET A   1    ' and lines[0][54:60] == '  1.00'
    assert np.allclose(xyz[0], [-24.430 + 1, 27.340 + 2, 2.614 - 300.5], atol=5e-4)


def test_checkpoint_dict_has_the_reference_keys(tmp_path):
    from equidock_public_b200.rigid_docking_model import Rigid_Body_Docking_Net
    args = gio.load_args('db5')
    args.update(device='cpu', worker=0, n_jobs=1, toy=False)
    model = Rigid_Body_Docking_Net(args)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    p = str(tmp_path / 'ck.pth')
    formats.save_checkpoint(p, model, opt.state_dict(), 7, args)
    a, sd, o, ep = formats.load_checkpoint(p)
    assert ep == 7 and set(sd) == set(model.state_dict()) and 'param_groups' in o
    assert all(k not in a for k in formats.NON_LOAD_KEYS) and a['iegmn_n_lays'] == args['iegmn_n_lays']
    Rigid_Body_Docking_Net({**a, 'device': 'cpu', 'debug': False}).load_state_dict(sd, strict=True)
