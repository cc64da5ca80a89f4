"""The oracle against outputs of the UNMODIFIED reference at full model sizes: every backbone at its default / BASELINE
configuration and every front-end configuration, recorded by tests/golden/make_golden.py in tests/golden/full_size.npz.
Weights and inputs are regenerated from the seeds in manifest.json.  Front-ends must match bit for bit everywhere;
embeddings bit for bit where the fixture was recorded and, on other CPUs, within 1e-6 plus the reference's own fp32-vs-fp64
gap (relative L2 per utterance)."""
import hashlib
import os

import numpy as np
import torch

from conftest import GOLDEN, rel_l2
from golden_data import arrays_sha256
from oracle import frontend as ofe
from oracle import models as om


def test_oracle_bit_level_against_reference_full_size(manifest):
    spec = manifest['full_size']
    z = np.load(os.path.join(GOLDEN, 'full_size.npz'))
    for i, (name, fdim, margs, B, T) in enumerate(spec['models']):
        sd = om.random_state_dict(name, fdim, seed=spec['weights_seed'], gain=om.CONDITIONED_GAIN[name], **margs)
        s = ';'.join(f'{k}:{tuple(v.shape)}' for k, v in sd.items())
        assert hashlib.sha256(s.encode()).hexdigest() == str(z[f'model{i}_params']), (name, margs)   # names, order, shapes
        x = torch.randn(B, T, fdim, generator=torch.Generator().manual_seed(spec['features_seed'])) * spec['features_scale']
        with torch.no_grad():
            emb = om.forward(name, sd, x, **margs).numpy()
        # bit for bit on the machine that recorded the fixture; elsewhere the CPU conv kernels sum in another order, so the
        # oracle may be no farther from the reference than the reference's fp32 result is from its own fp64 evaluation
        ref32, ref64 = z[f'model{i}_emb'], z[f'model{i}_emb64']
        err = rel_l2(emb, ref32)
        assert (err <= 1e-6 + rel_l2(ref32, ref64)).all(), (name, margs, err, rel_l2(ref32, ref64))

    w = torch.randn(*spec['wave_shape'], generator=torch.Generator().manual_seed(spec['wave_seed'])) * spec['wave_scale']
    ratio = torch.tensor(spec['ratio'])
    for j, (method, args) in enumerate(spec['front_ends']):
        assert ofe.feature_dim(method, args) == int(z[f'fe{j}_dim']), (method, args)
        for tag, out in (('batch', ofe.featurize(w, ratio, method, args)), ('single', ofe.featurize(w[1], None, method, args))):
            a = out.numpy()
            assert list(a.shape) == z[f'fe{j}_{tag}_shape'].tolist(), (method, args, tag)
            sample = a.ravel()[z[f'fe{j}_{tag}_idx']]
            assert np.array_equal(sample, z[f'fe{j}_{tag}_val']), (method, args, tag,
                                                                    np.abs(sample - z[f'fe{j}_{tag}_val']).max())
            assert arrays_sha256([('x', a)]) == str(z[f'fe{j}_{tag}_sha256']), (method, args, tag)   # bit exact
