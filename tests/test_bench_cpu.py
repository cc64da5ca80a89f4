"""CPU checks of the measurement harness: the synthetic workloads of bench.py are deterministic and identical in both
arms, the reference arm really drives the UNMODIFIED reference (oracle/_ref, installed by build()) in its own process, and the host-path chunk
planner cuts batches at wave boundaries."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_synthetic_workloads_are_deterministic_and_shared_by_both_arms():
    sys.path.insert(0, ROOT)
    import bench
    sys.path.insert(0, os.path.join(ROOT, 'baseline'))
    import ref_driver
    for name, cfg in bench.CONFIGS.items():
        lens = bench.batch_lens(cfg, 12, 99)
        assert lens == bench.batch_lens(cfg, 12, 99) and len(lens) == 12
        if cfg['ragged']:
            assert min(lens) >= 16000 and max(lens) <= 160000 and len(set(lens)) > 1
        else:
            assert set(lens) == {cfg['samples']}
    a = bench.synth_waves([1000, 700, 1300], 5)
    b = ref_driver.synth_waves([1000, 700, 1300], 5)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert abs(float(np.concatenate(a).std()) - 0.1) < 0.01


@pytest.mark.skipif(not os.path.isdir(os.path.join(ROOT, 'oracle', '_ref', 'mvector')),
                    reason='oracle/_ref not installed: build() found no checkout of the reference')
def test_reference_arm_runs_the_unmodified_reference():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--config', 'c2', '--steps', '1',
                        '--warmup', '1'], capture_output=True, text=True, timeout=600, cwd=ROOT,
                       env={k: v for k, v in os.environ.items() if k != 'PYTHONPATH'})
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])
    assert line['impl'] == 'reference' and line['value'] > 0 and line['unit'] == 'emb/s'
    assert line['cpu_baseline']['kind'] == 'reference' and line['cpu_baseline']['cores'] >= 1
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['gpu_launches'] == 0
    assert 'unmodified reference' in line['cpu_baseline']['sample']


def test_host_path_chunks_follow_wave_boundaries():
    sys.path.insert(0, ROOT)
    from mvector.predict import MVectorPredictor

    class P(MVectorPredictor):
        def __init__(self):
            pass

        def _chunk_size(self, B, T):
            return min(256, B)

    p = P()
    p.HOST_CHUNK = 128
    assert p._host_chunks(256, 298) == [127, 129]            # 127 x 298 rows = 296 tiles = two full waves of 148 SMs
    assert p._host_chunks(5, 298) == [5] and p._host_chunks(128, 298) == [128]
    for B, T in ((300, 298), (2048, 298), (700, 151), (64, 998)):
        c = p._host_chunks(B, T)
        assert sum(c) == B and all(0 < x <= 136 for x in c)
    p.HOST_CHUNK = 256
    assert p._host_chunks(256, 298) == [256] and p._host_chunks(600, 298)[0] in range(248, 257)
