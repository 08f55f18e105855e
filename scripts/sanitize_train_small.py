"""A small training step (forward with stash, device losses, CUDA backward, fused clip + Adam) for compute-sanitizer.
Optional argument: the dropout probability of the model (default 0: no dropout)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    sys.path.insert(0, p)
import numpy as np
import torch
import golden_io as gio
from equidock_public_b200 import hetero_graph as hg, synthetic
from equidock_public_b200.losses import PocketBatch
from equidock_public_b200.training import DataParallelTrainer
dev = torch.device('cuda:0')
rng = np.random.default_rng(0)
pairs = [synthetic.synthetic_pair(rng, a, b, 10) for a, b in ((70, 140), (129, 33))]
g = hg.batch_pairs(synthetic.to_torch_pairs(pairs)).to(dev)
bl = [torch.from_numpy(p[0]['x']) for p in pairs]
br = [torch.from_numpy(p[1]['x'] + 8.0) for p in pairs]
pk = [torch.from_numpy((0.5 * (p[0]['x'][:13] + p[1]['x'][:13] + 8.0)).astype(np.float32)) for p in pairs]
margs = dict(gio.load_args('db5'))
margs['dropout'] = float(sys.argv[1]) if len(sys.argv) > 1 else 0.0
tr = DataParallelTrainer(gio.build_model('db5', dev, args=margs), lr=1e-4)
out = tr.step(g, PocketBatch(bl, br, pk, pk, dev))
torch.cuda.synchronize()
print('done', float(out['loss'][0]))
