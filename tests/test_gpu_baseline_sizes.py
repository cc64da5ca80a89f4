"""GPU parity at the BASELINE.json sizes (SURVEY.md 8d), through the product API that bench.py times
(``MVectorPredictor.embed_device`` / ``predict_batch`` / ``mvector.distributed.predict_batch_sharded``):
every config at its full per-GPU batch, >= 16 utterances of it checked against the CPU oracle on the SAME padded batch
(identical waveforms, identical pad length -> identical per-utterance reference), plus the size-independent properties
(determinism, host-staged == device-resident bit for bit).  Tolerance: 1e-4 relative L2 (north_star)."""
import os
import socket
import tempfile

import numpy as np
import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu
EMB_TOL = 1e-4

FBANK80 = dict(sample_frequency=16000, num_mel_bins=80)
MEL64 = dict(sample_rate=16000, n_fft=1024, win_length=1024, hop_length=320, f_min=50.0, f_max=14000.0, n_mels=64)
CASES = {
    'c2': dict(model='EcapaTdnn', margs=dict(embd_dim=192, pooling_type='ASP', channels=[512, 512, 512, 512, 1536]),
               feature='Fbank', fargs=FBANK80, fdim=80, B=256, lens=lambda g: [48000] * 256),
    'c3': dict(model='CAMPPlus', margs=dict(embd_dim=192), feature='Fbank', fargs=FBANK80, fdim=80, B=256,
               lens=lambda g: [48000] * 256),
    'c4': dict(model='ResNetSE', margs=dict(embd_dim=192, pooling_type='ASP'), feature='MelSpectrogram', fargs=MEL64, fdim=64,
               B=128, lens=lambda g: [80000] * 128),
    # ragged 1-10 s; item 0 is pinned to 10 s so that T = 998 (K = 9216 chunked accumulation at its longest M) always runs
    'c5': dict(model='ERes2Net', margs=dict(embd_dim=192, m_channels=64, mul_channel=2, expansion=4, base_width=24, scale=3),
               feature='Fbank', fargs=FBANK80, fdim=80, B=64,
               lens=lambda g: [160000] + torch.randint(16000, 160001, (63,), generator=g).tolist()),
}


def _cfg(c):
    return {'dataset_conf': {'dataset': {'min_duration': 0.3, 'max_duration': 3, 'sample_rate': 16000,
                                         'use_dB_normalization': False, 'target_dB': -20},
                             'eval_conf': {'batch_size': 16, 'max_duration': 20}},
            'preprocess_conf': {'use_hf_model': False, 'feature_method': c['feature'], 'method_args': dict(c['fargs'])},
            'model_conf': {'model': c['model'], 'model_args': dict(c['margs'])}}


def _predictor(c, sd):
    from loguru import logger
    logger.remove()
    from mvector.predict import MVectorPredictor
    with tempfile.TemporaryDirectory() as td:
        torch.save({'0.' + k: v for k, v in sd.items()}, os.path.join(td, 'model.pth'))
        return MVectorPredictor(configs=_cfg(c), model_path=td, use_gpu=True)


def _weights(c, seed=0):
    from oracle import models as om
    gain = om.CONDITIONED_GAIN.get(c['model']) if hasattr(om, 'CONDITIONED_GAIN') else None
    kw = dict(gain=gain) if gain is not None else {}
    return om.random_state_dict(c['model'], c['fdim'], seed=seed, **kw, **c['margs'])


@pytest.mark.parametrize('name', ['c2', 'c3', 'c4', 'c5'])
def test_baseline_config_full_batch_vs_oracle(name):
    import warnings
    from oracle import frontend as ofe
    from oracle import models as om
    c = CASES[name]
    g = torch.Generator().manual_seed(100 + ord(name[1]))
    lens = c['lens'](g)
    B, lmax = c['B'], max(lens)
    waves = [(torch.randn(n, generator=g) * 0.1).numpy() for n in lens]
    sd = _weights(c)
    pred = _predictor(c, sd)
    # (1) the public API on host data (native staging pipeline), (2) the device-resident path bench.py's `value` times
    e_host = pred.predict_batch(waves)
    assert e_host.shape == (B, 192) and e_host.dtype == np.float32 and np.isfinite(e_host).all()
    x = np.zeros((B, lmax), dtype=np.float32)
    for i, w in enumerate(waves):
        x[i, :w.shape[0]] = w
    xd = torch.from_numpy(x).cuda()
    e_dev = pred.embed_device(xd, lens)
    assert torch.equal(pred.embed_device(xd, lens), e_dev)                   # deterministic (no float atomics on the path)
    into = torch.empty_like(e_dev)
    assert pred.embed_device(xd, lens, out=into) is into and torch.equal(into, e_dev)   # caller-owned output rows
    # host-staged vs device-resident: the same kernels on the same data.  With the same backbone chunking they agree bit
    # for bit; the default host path uses smaller chunks (to overlap staging with compute), and a chunk's fp16-split
    # activation scale is a property of the tensor the kernel sees, so the default agrees to a few ulp (DESIGN 4.1)
    assert rel_l2(e_host, e_dev.cpu().numpy()).max() <= 2e-6
    pred.HOST_CHUNK = pred.MAX_BATCH
    assert np.array_equal(pred.predict_batch(waves), e_dev.cpu().numpy())
    del pred.HOST_CHUNK
    # (3) >= 16 utterances against the CPU oracle on the same padded batch (first / last / longest / shortest / spread)
    idx = sorted(set([0, B - 1, int(np.argmax(lens)), int(np.argmin(lens))] + list(range(3, B, max(B // 14, 1)))))[:18]
    assert len(idx) >= 16
    ratio = torch.tensor([lens[i] / lmax for i in idx], dtype=torch.float32)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        feats = ofe.featurize(torch.from_numpy(x[idx]), ratio, c['feature'], c['fargs'])
    ref = om.forward(c['model'], sd, feats, **c['margs']).numpy()
    err = rel_l2(e_host[idx], ref)
    print(f'{name}: B={B} Lmax={lmax} T={feats.shape[1]} sampled {len(idx)} utterances, max rel-L2 {err.max():.2e}')
    assert err.max() < EMB_TOL, (name, err)


def test_program_cache_shares_one_workspace_arena():
    """Ragged serving: programs of different (B, T) share the handle's arena (max, not sum, of their workspaces) and
    revisiting a shape after others ran gives bit-identical results."""
    from mvector import _lib as L
    c = CASES['c2']
    sd = _weights(c, seed=4)
    pred = _predictor(c, sd)
    g = torch.Generator().manual_seed(3)
    outs = {}
    sizes = []
    for T in (120, 298, 77, 500, 298, 120):
        f = torch.randn(4, T, 80, generator=g).cuda() if T not in outs else outs[T][0]
        e = pred.predictor(f)
        if T in outs:
            assert torch.equal(e, outs[T][1]), T
        outs[T] = (f, e.clone())
        sizes.append(int(L.lib().vp_workspace_bytes(pred._engine.handle)))
    assert sizes == sorted(sizes), sizes                                     # the arena only grows
    ws = [pred.predictor.program(4, T).ws_bytes for T in (120, 298, 77, 500)]
    assert max(ws) <= sizes[-1] < sum(ws)


def test_embed_wave_rejects_mismatched_call_before_launching():
    """ADVICE r1: vp_embed_wave must validate (B, Lpad) against the program before the front-end writes anything."""
    import ctypes as C
    from mvector import _lib as L
    c = CASES['c2']
    pred = _predictor(c, _weights(c, seed=5))
    fz = pred._audio_featurizer
    T = fz.num_frames(16000)
    prog = pred.predictor.program(2, T)
    wave = torch.zeros(3, 16000, device='cuda')
    feats = torch.full((2 * T * 80,), 7.0, device='cuda')                    # sized from the PROGRAM (2 utterances)
    scratch = torch.zeros(int(L.lib().vp_frontend_scratch_floats(fz.engine.handle, 3, 16000)), device='cuda')
    emb = torch.zeros(2, 192, device='cuda')
    with pytest.raises(L.VpError):
        prog.run_wave(wave, None, feats, scratch, emb)                       # B = 3 against a B = 2 program
    with pytest.raises(L.VpError):
        prog.run_wave(wave[:2, :8000].contiguous(), None, feats, scratch, emb)   # right B, wrong length
    torch.cuda.synchronize()
    assert bool((feats == 7.0).all())                                        # nothing was launched


# ------------------------------------------------------------------------------------------------ sharded product path
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_worker(rank, world, port, backend, feature, same_gpu, out_dir):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dev = 0 if same_gpu else rank
    torch.cuda.set_device(dev)
    if backend == 'nccl':
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', dev))
    else:
        dist.init_process_group('gloo', rank=rank, world_size=world)
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, 'tests')):
        if p not in sys.path:
            sys.path.insert(0, p)
    from mvector.distributed import predict_batch_sharded
    c = dict(CASES['c2'])
    c['margs'] = dict(embd_dim=192, pooling_type='ASP', channels=[128, 128, 128, 128, 384], attention_channels=64,
                      res2net_scale=4, se_channels=32)
    if feature == 'MFCC':                   # the one front-end with a cross-utterance term (call-wide top_db clamp)
        c['feature'], c['fargs'], c['fdim'] = 'MFCC', dict(n_mfcc=40), 40
    sd = _weights(c, seed=9)
    pred = _predictor(c, sd)
    g = torch.Generator().manual_seed(77)                                    # identical list on every rank
    lens = [16000, 48000, 30001, 5000, 160000, 21000, 64000, 8000, 100000]   # 9 items -> uneven shards, ragged 0.3-10 s
    amp = [0.1, 0.3, 0.1, 1e-4, 0.1, 0.05, 0.2, 0.1, 0.1]                     # a quiet item: clamped by the OTHER rank's max
    waves = [(torch.randn(n, generator=g) * a).numpy() for n, a in zip(lens, amp)]
    full = pred.predict_batch(waves)                                         # single-process reference semantics
    got = predict_batch_sharded(pred, waves)
    np.save(os.path.join(out_dir, f'rank{rank}.npy'), np.stack([full, got]))
    dist.barrier()
    dist.destroy_process_group()


def _run_sharded(world, backend, feature, same_gpu):
    """Sharded vs single-process result of the same list, on every rank.

    * split-TF32 engine (VPB_TC_F16=0): BIT EXACT -- every op is per-utterance and shard-invariant (global Lmax padding,
      MFCC's call-wide clamp maximum all-reduced), so sharding cannot change a single bit.
    * default engine (two-term FP16 split): the power-of-two activation scale of a layer comes from the maximum over the
      tensor the kernel sees -- the whole batch in one process, the shard under sharding.  A different power of two moves
      the fp16 subnormal floor of the lo terms (relative 2^-38 of the tensor maximum), which can flip the last bit of an
      fp32 accumulation: agreement to a few ulp (<= 2e-6 relative L2), not bit for bit."""
    import torch.multiprocessing as mp
    for f16, tol in (('0', 0.0), ('1', 2e-6)):
        old = os.environ.get('VPB_TC_F16')
        os.environ['VPB_TC_F16'] = f16                  # read at library load in the spawned ranks
        try:
            with tempfile.TemporaryDirectory() as td:
                mp.spawn(_sharded_worker, args=(world, _free_port(), backend, feature, same_gpu, td), nprocs=world, join=True)
                for r in range(world):
                    full, got = np.load(os.path.join(td, f'rank{r}.npy'))
                    assert got.shape == (9, 192)
                    if tol == 0.0:
                        assert np.array_equal(full, got), (feature, r, np.abs(full - got).max())
                    else:
                        assert rel_l2(got, full).max() <= tol, (feature, r, rel_l2(got, full).max())
        finally:
            if old is None:
                os.environ.pop('VPB_TC_F16', None)
            else:
                os.environ['VPB_TC_F16'] = old


@pytest.mark.parametrize('feature', ['Fbank', 'MFCC'])
def test_predict_batch_sharded_two_ranks_one_gpu(feature):
    """The product sharding API on real kernels when the box has ONE GPU: two processes share cuda:0, collectives over
    gloo (NCCL refuses two ranks on one device).  Ragged batch -> global Lmax padding; MFCC -> all-reduce(MAX)."""
    _run_sharded(2, 'gloo', feature, same_gpu=True)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
@pytest.mark.parametrize('feature', ['Fbank', 'MFCC'])
def test_predict_batch_sharded_nccl_two_gpus(feature):
    """One process per GPU over NCCL: the sharded result equals the single-process predict_batch bit for bit."""
    _run_sharded(2, 'nccl', feature, same_gpu=False)
