#!/usr/bin/env python
"""Reference arm of bench.py: times the UNMODIFIED reference (yeyupiaoling/VoiceprintRecognition-Pytorch, mvector 1.1.1,
installed into oracle/_ref by build(), oracle/reference.py) through its OWN public API --
``mvector.predict.MVectorPredictor(configs, model_path, use_gpu).predict_batch(list of numpy waveforms)``
(predict.py:231-265) -- on the box's host cores (``--device cpu``) or, for the same-box GPU-library bar, on cuda with the
stock PyTorch eager kernels (cuDNN / cuBLAS; ``--device cuda``).  None of this repo's code is on that path.

The one thing that cannot come from the reference tree is its third-party dependency ``yeaudio`` (requirements.txt:12,
absent from the image): ``predict.py:13`` imports ``yeaudio.audio.AudioSegment`` and ``_load_audio`` calls
``AudioSegment.from_ndarray`` on every waveform (predict.py:192-199).  A ~20-line stand-in provides exactly that
constructor (fields ``samples / sample_rate / duration``); no arithmetic of the timed path lives in it.

Run as a separate process (``python baseline/ref_driver.py spec.json``) from bench.py so that the reference's package
``mvector`` never meets this repo's package of the same name.  Prints ONE JSON line."""
import json
import os
import sys
import time
import types

HERE = os.path.dirname(os.path.abspath(__file__))


def _install_yeaudio_stub():
    import numpy as np

    class AudioSegment:
        def __init__(self, samples, sample_rate):
            self.samples = np.asarray(samples, dtype=np.float32)
            self.sample_rate = sample_rate

        @property
        def duration(self):
            return self.samples.shape[0] / float(self.sample_rate)

        @classmethod
        def from_ndarray(cls, data, sample_rate=16000):
            return cls(data, sample_rate)

        def resample(self, sr):
            raise NotImplementedError('bench waveforms are already at the target rate')

        def normalize(self, target_db=-20, max_gain_db=300.0):
            raise NotImplementedError('bench configs run with use_dB_normalization=False')

    mod, sub = types.ModuleType('yeaudio'), types.ModuleType('yeaudio.audio')
    sub.AudioSegment = AudioSegment
    mod.audio = sub
    sys.modules['yeaudio'], sys.modules['yeaudio.audio'] = mod, sub


def synth_waves(lens, seed):
    """Same generator as bench.py: one seeded randn stream, sigma 0.1 (= -20 dBFS), utterance i takes lens[i] samples."""
    import torch
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(int(n), generator=g) * 0.1).numpy() for n in lens]


def main():
    spec = json.load(open(sys.argv[1]))
    ref_root = spec.get('ref_root') or os.path.join(os.path.dirname(HERE), 'oracle', '_ref')
    if not os.path.isdir(os.path.join(ref_root, 'mvector')):
        print(json.dumps({'unavailable': f'no reference install at {ref_root}'}))
        return
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or '.') != os.path.dirname(HERE)]   # keep this repo's `mvector` out
    sys.path.insert(0, ref_root)
    device = spec.get('device', 'cpu')
    if device == 'cpu' and spec.get('threads'):
        os.environ['OMP_NUM_THREADS'] = str(spec['threads'])
    import numpy as np
    import torch
    from loguru import logger
    logger.remove()
    _install_yeaudio_stub()
    from mvector.predict import MVectorPredictor          # the reference's own class, unmodified
    import mvector
    assert os.path.abspath(mvector.__file__).startswith(os.path.abspath(ref_root)), mvector.__file__

    if device == 'cuda':
        tf32 = spec.get('tf32')                            # None = PyTorch defaults (cuDNN conv TF32 on, matmul TF32 off)
        if tf32 is not None:
            torch.backends.cudnn.allow_tf32 = bool(tf32)
            torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    cfg = spec['configs']
    pred = MVectorPredictor(configs=cfg, model_path=spec['model_path'], use_gpu=(device == 'cuda'))
    waves = synth_waves(spec['lens'], spec['seed'])

    mode = spec.get('mode', 'predict_batch')
    if mode == 'predict_batch':
        def one_pass():
            return pred.predict_batch(waves, sample_rate=16000)   # default batch_size=32 (predict.py:231)
    else:
        # 'model_only': the reference's modules with the features already resident on the device -- the most favourable
        # reading of "PyTorch eager on the same GPU" (predict_batch itself runs the Kaldi front-end on the CPU,
        # predict.py:256).  Same chunk loop as predict.py:259-262 with batch_size from the spec.
        lmax = max(w.shape[0] for w in waves)
        x = np.zeros((len(waves), lmax), dtype=np.float32)
        for i, w in enumerate(waves):
            x[i, :w.shape[0]] = w
        ratio = torch.tensor([w.shape[0] / lmax for w in waves], dtype=torch.float32)
        feats = pred._audio_featurizer(torch.tensor(x), ratio).to(pred.device)
        bs = int(spec.get('batch_size', 32))

        def one_pass():
            out = []
            with torch.no_grad():
                for i in range(0, feats.shape[0], bs):
                    out.extend(pred.predictor(feats[i:i + bs]).data.cpu().numpy())
            return np.array(out)

    threads = None
    if device == 'cpu':
        # torchrun pins OMP_NUM_THREADS=1 and an oversubscribed host is slower with every hardware thread: try the whole
        # machine, half and a quarter on a short probe and keep the fastest (= the strongest CPU baseline)
        ncpu = os.cpu_count() or 1
        cands = [int(spec['threads'])] if spec.get('threads') else sorted({ncpu, max(ncpu // 2, 1), max(ncpu // 4, 1)}, reverse=True)
        probe = waves[:max(2, min(len(waves), 8))]
        best = None
        for n in cands:
            torch.set_num_threads(n)
            pred.predict_batch(probe)
            t0 = time.perf_counter()
            pred.predict_batch(probe)
            t = time.perf_counter() - t0
            if best is None or t < best[1]:
                best = (n, t)
        threads = best[0]
        torch.set_num_threads(threads)
    sync = (lambda: torch.cuda.synchronize()) if device == 'cuda' else (lambda: None)
    emb = None
    for _ in range(int(spec.get('warmup', 1))):
        emb = one_pass()
    sync()
    steps = int(spec.get('steps', 1))
    budget = float(spec.get('budget_s', 0))
    done, t0 = 0, time.perf_counter()
    while True:
        emb = one_pass()
        done += 1
        sync()
        el = time.perf_counter() - t0
        if done >= steps and el >= budget:
            break
    out = {'emb_per_s': len(waves) * done / el, 'ms_per_step': 1e3 * el / done, 'steps': done, 'n_utts': len(waves),
           'elapsed_s': el, 'device': device, 'threads': threads, 'torch': torch.__version__, 'mode': mode,
           'api': 'mvector.predict.MVectorPredictor.predict_batch (unmodified reference, oracle/_ref)'}
    if device == 'cuda':
        out['tf32'] = {'cudnn': torch.backends.cudnn.allow_tf32, 'matmul': torch.backends.cuda.matmul.allow_tf32}
        out['gpu'] = torch.cuda.get_device_name(0)
    else:
        try:
            with open('/proc/cpuinfo') as f:
                out['cpu_model'] = next(l.split(':', 1)[1].strip() for l in f if l.startswith('model name'))
        except Exception:
            out['cpu_model'] = None
    if spec.get('save_emb'):
        np.save(spec['save_emb'], np.asarray(emb, dtype=np.float32))
    print(json.dumps(out))


if __name__ == '__main__':
    main()
