"""Host-side logic that needs no GPU: C-ABI library loads and exports every symbol of include/vpb200.h, the tensor-core
weight image packer, front-end constants, config surface, audio decoding, memory planner."""
import ctypes
import io
import os
import re
import wave

import numpy as np
import pytest
import torch

from golden_data import arrays_sha256, diarization_vad

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    lib_path = ge.build()
    hdr = open(os.path.join(ROOT, 'include', 'vpb200.h')).read()
    declared = set(re.findall(r'\b(vp_[a-z_0-9]+)\s*\(', hdr))
    assert len(declared) >= 18
    lib = ctypes.CDLL(lib_path)
    for name in sorted(declared):
        assert hasattr(lib, name), f'{name} declared in vpb200.h but not exported by libvpb200.so'
    from mvector import _lib
    assert set(_lib.EXPORTS) == declared
    L = _lib.lib()
    assert L.vp_abi_version() == 4
    assert L.vp_sizeof_op() == ctypes.sizeof(_lib.Op)


def test_no_gpu_means_loud_failure_not_fallback():
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from mvector.engine import Engine
    from mvector.predict import MVectorPredictor
    with pytest.raises(RuntimeError):
        Engine()
    with pytest.raises(AssertionError):
        MVectorPredictor(configs={}, use_gpu=True)


def test_pack_tc_image_roundtrip():
    """Split-TF32 weight image: hi has a 10-bit mantissa, hi + lo == W exactly, and un-swizzling the SWIZZLE_128B
    chunk permutation gives back the zero-padded [n_tile][k_block][BN][32] tiles."""
    from mvector.engine import pack_tc, tc_tile_n, tf32_rna
    rng = np.random.default_rng(0)
    for N, K in ((512, 512), (192, 400), (128, 1536), (32, 384), (24, 72), (512, 2304)):
        W = rng.standard_normal((N, K)).astype(np.float32)
        img, bn = pack_tc(W.astype(np.float64))
        assert bn == tc_tile_n(N, K > 1536) and bn % 16 == 0 and bn <= 256
        nt, kb = -(-N // bn), -(-K // 32)
        t = img.reshape(nt, kb, 2, bn, 8, 4)
        r = np.arange(bn)[:, None]
        c = np.arange(8)[None, :]
        un = t[:, :, :, r, c ^ (r & 7), :]                      # undo the XOR swizzle
        un = un.reshape(nt, kb, 2, bn, 32)
        hi = un[:, :, 0].transpose(0, 2, 1, 3).reshape(nt * bn, kb * 32)
        lo = un[:, :, 1].transpose(0, 2, 1, 3).reshape(nt * bn, kb * 32)
        assert np.array_equal(hi[:N, :K] + lo[:N, :K], W)
        assert not (hi.view(np.uint32) & 0x1FFF).any()
        assert np.all(hi[N:] == 0) and np.all(hi[:, K:] == 0) and np.all(lo[N:] == 0)
        assert np.abs(lo[:N, :K]).max() <= np.abs(W).max() * 2.0 ** -11 * 1.01
    x = np.float32([1.0 + 2.0 ** -11, 1.0 + 2.0 ** -11 + 2.0 ** -20, -(1.0 + 2.0 ** -11)])
    assert np.array_equal(tf32_rna(x), np.float32([1.0 + 2.0 ** -10, 1.0 + 2.0 ** -10, -(1.0 + 2.0 ** -10)]))  # ties away


def test_frontend_constants_match_oracle():
    from mvector.data_utils.featurizer import KaldiFbank, MelSpectrogram
    from oracle import frontend as ofe
    kf = KaldiFbank(sample_frequency=16000, num_mel_bins=80)
    assert (kf.n_fft, kf.win_length, kf.hop, kf.n_mels) == (512, 400, 160, 80)
    assert np.array_equal(kf.window, ofe.feature_window('povey', 400).numpy())
    dense = torch.nn.functional.pad(ofe.kaldi_mel_banks(80, 512, 16000.0, 20.0, 0.0), (0, 1)).numpy()
    start, count, off, w = kf.bank
    rec = np.zeros_like(dense)
    for m in range(80):
        rec[m, start[m]:start[m] + count[m]] = w[off[m]:off[m] + count[m]]
    assert np.array_equal(rec, dense)
    assert int(count.sum()) < 600                       # ~501 non-zeros (SURVEY.md 9.1)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        ms = MelSpectrogram(sample_rate=16000, n_fft=1024, win_length=1024, hop_length=320, f_min=50.0, f_max=14000.0,
                            n_mels=64)
    fb = ofe.htk_mel_fbanks(513, 50.0, 14000.0, 64, 16000).numpy().T
    start, count, off, w = ms.bank
    rec = np.zeros_like(fb)
    for m in range(64):
        rec[m, start[m]:start[m] + count[m]] = w[off[m]:off[m] + count[m]]
    assert np.array_equal(rec, fb)


def test_featurizer_surface():
    from mvector.data_utils.featurizer import AudioFeaturizer
    fz = AudioFeaturizer('Fbank', method_args=dict(sample_frequency=16000, num_mel_bins=80))
    assert fz.feature_dim == 80 and fz.num_frames(48000) == 298 and fz.num_frames(399) == 0
    assert AudioFeaturizer('MelSpectrogram', method_args=dict(n_fft=512, n_mels=40)).feature_dim == 40
    # mask_lens = round(ratio * T) in float32, half to even (featurizer.py:82-84)
    assert fz.keep_frames([16000 / 48000, 1.0, 0.5], 298).tolist() == [99, 298, 149]
    assert fz.keep_frames([0.5], 297).tolist() == [148]
    with pytest.raises(TypeError):
        AudioFeaturizer('Fbank', method_args=dict(bogus=1))
    # torchaudio defaults (n_fft = 400, a 2^4 5^2 FFT) are accepted for all three STFT front-ends
    assert AudioFeaturizer('MFCC').feature_dim == 40 and AudioFeaturizer('Spectrogram').feature_dim == 201
    assert AudioFeaturizer('MelSpectrogram').feature_dim == 128
    assert AudioFeaturizer('Spectrogram', method_args=dict(n_fft=512)).num_frames(16000) == 1 + 16000 // 256
    with pytest.raises(NotImplementedError):
        AudioFeaturizer('Spectrogram', method_args=dict(n_fft=442))          # 442 = 2 * 13 * 17
    with pytest.raises(ValueError):
        AudioFeaturizer('MFCC', method_args=dict(n_mfcc=200))
    with pytest.raises(NotImplementedError):
        AudioFeaturizer('Fbank', use_hf_model=True)
    with pytest.raises(Exception):
        AudioFeaturizer('Nope')


def test_audio_segment_wav_and_normalize():
    from mvector.audio import AudioSegment
    pcm = (np.sin(np.arange(16000) * 0.05) * 8000).astype('<i2')
    buf = io.BytesIO()
    with wave.open(buf, 'wb') as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000); w.writeframes(pcm.tobytes())
    seg = AudioSegment.from_bytes(buf.getvalue())
    assert seg.sample_rate == 16000 and abs(seg.duration - 1.0) < 1e-9
    assert np.array_equal(seg.samples, pcm.astype(np.float32) / 32768.0)
    seg.normalize(target_db=-20)
    assert abs(seg.rms_db - (-20)) < 1e-3
    seg.resample(8000)
    assert seg.sample_rate == 8000 and abs(seg.samples.shape[0] - 8000) <= 1


def test_memory_planner_reuses_and_never_overlaps_live_buffers():
    from mvector.engine import PlanBuilder
    pb = PlanBuilder(1)
    live = {}
    rng = np.random.default_rng(1)
    for step in range(300):
        if live and rng.random() < 0.45:
            k = list(live)[rng.integers(len(live))]
            pb.free(live.pop(k))
        else:
            v = pb.alloc(int(rng.integers(1, 2000)), int(rng.integers(1, 64)) * 4)
            live[v.off] = v
        iv = sorted((v.off, v.off + pb._live[v.off]) for v in live.values())
        for (a0, a1), (b0, b1) in zip(iv, iv[1:]):
            assert a1 <= b0
        assert all(e <= pb.peak for _, e in iv)
    assert pb.peak < 300 * 2000 * 256 * 4 / 4            # reuse happened


def test_default_model_plans_lower_and_fit(manifest):
    """Every BASELINE configuration lowers on the host; report op counts / workspace."""
    from mvector.models import build_model
    from mvector.utils.utils import dict_to_object
    from oracle import models as om
    cases = [('EcapaTdnn', 80, dict(embd_dim=192, pooling_type='ASP', channels=[512, 512, 512, 512, 1536]), 256, 298),
             ('CAMPPlus', 80, dict(embd_dim=192), 256, 298),
             ('TDNN', 80, dict(embd_dim=192, channels=512, pooling_type='ASP'), 1, 365)]
    for name, fdim, margs, B, T in cases:
        m = build_model(fdim, dict_to_object({'model_conf': {'model': name, 'model_args': margs}}))
        m.load_state_dict(om.random_state_dict(name, fdim, seed=0, **margs))
        pb = m.lower(B, T)
        assert pb.in_floats == B * T * fdim and pb.out_floats == B * 192
        assert pb.peak < 40 * 2 ** 30


def test_host_gather_pad_native():
    """vp_host_gather_pad: the zero-padded [n, lmax] staging matrix of predict.py:248-254, multi-threaded, no GPU."""
    import ctypes as C
    from mvector import _lib as L
    rng = np.random.default_rng(3)
    lens = [int(x) for x in rng.integers(1, 5000, size=37)] + [5000]
    ws = [rng.standard_normal(n).astype(np.float32) for n in lens]
    lmax = max(lens)
    dst = np.full((len(ws), lmax), np.nan, dtype=np.float32)
    ptrs = (C.c_void_p * len(ws))(*[w.ctypes.data for w in ws])
    ln = (C.c_int32 * len(ws))(*lens)
    for threads in (1, 4):
        dst[:] = np.nan
        assert L.lib().vp_host_gather_pad(ptrs, ln, len(ws), lmax, dst.ctypes.data_as(C.c_void_p), threads) == 0
        for i, w in enumerate(ws):
            assert np.array_equal(dst[i, :len(w)], w) and not dst[i, len(w):].any()
    bad = (C.c_int32 * len(ws))(*([lmax + 1] + lens[1:]))
    assert L.lib().vp_host_gather_pad(ptrs, bad, len(ws), lmax, dst.ctypes.data_as(C.c_void_p), 2) == L.VP_ERR_INVALID


def test_host_stage_pool_reuse_slices_and_threads():
    """vp_host_stage_h2d without a device target (gather only, no CUDA call): every slice / thread split gives the same
    staging matrix, back-to-back jobs reuse the persistent worker pool, and a numpy-uint64 pointer table (what
    predict_batch passes) is accepted."""
    import ctypes as C
    from mvector import _lib as L
    rng = np.random.default_rng(5)
    lens = np.asarray([int(x) for x in rng.integers(1, 3000, size=101)], dtype=np.int32)
    ws = [rng.standard_normal(int(n)).astype(np.float32) for n in lens]
    lmax = int(lens.max())
    ref = np.zeros((len(ws), lmax), dtype=np.float32)
    for i, w in enumerate(ws):
        ref[i, :len(w)] = w
    ptrs = np.fromiter((w.__array_interface__['data'][0] for w in ws), dtype=np.uint64, count=len(ws))
    for rep in range(3):
        for slice_rows, threads in ((1, 8), (7, 3), (16, 2), (101, 1), (200, 4), (5, 32)):
            dst = np.full((len(ws), lmax), np.nan, dtype=np.float32)
            rc = L.lib().vp_host_stage_h2d(C.c_void_p(ptrs.ctypes.data), C.c_void_p(lens.ctypes.data), len(ws), lmax,
                                           dst.ctypes.data_as(C.c_void_p), C.c_void_p(), slice_rows, threads, C.c_void_p())
            assert rc == 0 and np.array_equal(dst, ref), (rep, slice_rows, threads)
    # a sub-range of the list (what a staging call of predict_batch passes): rows 40..60
    dst = np.full((20, lmax), np.nan, dtype=np.float32)
    rc = L.lib().vp_host_stage_h2d(C.c_void_p(ptrs.ctypes.data + 8 * 40), C.c_void_p(lens.ctypes.data + 4 * 40), 20, lmax,
                                   dst.ctypes.data_as(C.c_void_p), C.c_void_p(), 4, 3, C.c_void_p())
    assert rc == 0 and np.array_equal(dst, ref[40:60])
    assert L.lib().vp_host_stage_h2d(C.c_void_p(ptrs.ctypes.data), C.c_void_p(lens.ctypes.data), len(ws), lmax,
                                     dst.ctypes.data_as(C.c_void_p), C.c_void_p(), 0, 2, C.c_void_p()) == L.VP_ERR_INVALID


def test_host_stage_copy_path_with_stub_runtime(tmp_path):
    """The copy-issuing half of vp_host_stage_h2d without a GPU: host_util.cu + host_copy.cpp compiled with g++ against a
    test double of cuda_runtime.h (tests/stubs: "device" = host memory, cudaMemcpyAsync = memcpy + log).  The copies must
    tile [0, n * lmax) in order without gaps or overlap (consecutive finished slices may be merged into one copy), the
    "device" matrix must equal the zero-padded reference for every thread count / slice size / store mode, and a failing
    copy is reported as VP_ERR_CUDA after the job has drained."""
    import ctypes as C
    import subprocess
    csrc = os.path.join(ROOT, 'voiceprintrecognition-pytorch_b200', 'csrc')
    so = str(tmp_path / 'libstage_stub.so')
    cmd = ['g++', '-O2', '-std=c++17', '-shared', '-fPIC', '-pthread', '-I', os.path.join(ROOT, 'tests', 'stubs'),
           '-x', 'c++', os.path.join(csrc, 'host_util.cu'), os.path.join(csrc, 'host_copy.cpp'),
           os.path.join(ROOT, 'tests', 'stubs', 'stub_runtime.cpp'), '-o', so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(so)
    lib.vp_host_stage_h2d.restype = C.c_int
    lib.vp_host_stage_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_void_p]
    lib.stub_get.argtypes = [C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    rng = np.random.default_rng(3)
    for trial in range(8):
        n, lmax = int(rng.integers(1, 150)), int(rng.integers(1, 5000))
        lens = rng.integers(0, lmax + 1, n).astype(np.int32)
        lens[int(rng.integers(0, n))] = lmax
        ws = [rng.standard_normal(max(int(ln), 1)).astype(np.float32) for ln in lens]
        ptrs = np.fromiter((w.__array_interface__['data'][0] for w in ws), dtype=np.uint64, count=n)
        ref = np.zeros((n, lmax), dtype=np.float32)
        for i, w in enumerate(ws):
            ref[i, :lens[i]] = w[:lens[i]]
        for streaming in (0, 1):
            lib.vp_host_gather_streaming(streaming)
            for threads, slice_rows in ((1, 1), (1, 7), (2, 4), (8, 4), (8, 1), (4, 1000)):
                staging = np.full((n, lmax), np.nan, dtype=np.float32)
                device = np.full((n, lmax), np.nan, dtype=np.float32)
                lib.stub_reset(C.c_void_p(device.ctypes.data), -1)
                rc = lib.vp_host_stage_h2d(ptrs.ctypes.data, lens.ctypes.data, n, lmax, staging.ctypes.data, device.ctypes.data,
                                           slice_rows, threads, None)
                assert rc == 0 and np.array_equal(device, ref) and np.array_equal(staging, ref), (trial, threads, slice_rows)
                pos, n_slices = 0, (n + slice_rows - 1) // slice_rows
                assert 1 <= lib.stub_count() <= n_slices
                for k in range(lib.stub_count()):
                    off, nb = C.c_size_t(), C.c_size_t()
                    lib.stub_get(k, C.byref(off), C.byref(nb))
                    assert off.value == pos and nb.value > 0 and nb.value % (4 * lmax) == 0   # whole rows, in order, no gap
                    assert (nb.value // (4 * lmax)) % slice_rows == 0 or pos + nb.value == n * lmax * 4
                    pos += nb.value
                assert pos == n * lmax * 4
        # a copy that fails: error code after the job has drained, no hang, later calls work again
        device = np.zeros((n, lmax), dtype=np.float32)
        staging = np.zeros((n, lmax), dtype=np.float32)
        lib.stub_reset(C.c_void_p(device.ctypes.data), 0)
        assert lib.vp_host_stage_h2d(ptrs.ctypes.data, lens.ctypes.data, n, lmax, staging.ctypes.data, device.ctypes.data,
                                     2, 3, None) == 2                  # VP_ERR_CUDA
        assert np.array_equal(staging, ref)
    lib.vp_host_gather_streaming(0)


def test_host_stage_streaming_stores_same_bytes():
    """vp_host_gather_streaming(1): the gather writes the pinned rows with non-temporal stores (AVX2 / AVX-512 picked at run
    time).  Same staging matrix as memcpy for every alignment of source and destination, nothing written outside the
    matrix, and the switch reports whether streaming stores are in effect."""
    import ctypes as C
    from mvector import _lib as L
    lib = L.lib()
    try:
        eff = lib.vp_host_gather_streaming(1)
        assert eff in (0, 1) and lib.vp_host_gather_streaming(-1) == eff
        rng = np.random.default_rng(11)
        for trial in range(12):
            n, lmax = int(rng.integers(1, 60)), int(rng.integers(1, 9000))
            lens = rng.integers(0, lmax + 1, n).astype(np.int32)
            lens[int(rng.integers(0, n))] = lmax
            ws = []
            for ln in lens:                              # sources at odd float offsets inside their allocations
                off = int(rng.integers(0, 17))
                base = rng.standard_normal(int(ln) + off + 1).astype(np.float32)
                ws.append(base[off:off + int(ln)] if ln > 0 else base[:1])
            ptrs = np.fromiter((w.__array_interface__['data'][0] for w in ws), dtype=np.uint64, count=n)
            ref = np.zeros((n, lmax), dtype=np.float32)
            for i, w in enumerate(ws):
                ref[i, :lens[i]] = w[:lens[i]]
            for threads, slice_rows in ((1, 1), (2, 4), (8, 3), (3, 100)):
                o = int(rng.integers(0, 16))             # destination at every 4-byte phase of a cache line
                buf = np.full(n * lmax + 16, 7.0, dtype=np.float32)
                dst = buf[o:o + n * lmax].reshape(n, lmax)
                rc = lib.vp_host_stage_h2d(C.c_void_p(ptrs.ctypes.data), C.c_void_p(lens.ctypes.data), n, lmax,
                                           C.c_void_p(dst.ctypes.data), C.c_void_p(), slice_rows, threads, C.c_void_p())
                assert rc == 0 and np.array_equal(dst, ref), (trial, threads, slice_rows)
                assert (buf[:o] == 7.0).all() and (buf[o + n * lmax:] == 7.0).all()
    finally:
        lib.vp_host_gather_streaming(0)
    assert lib.vp_host_gather_streaming(-1) == 0


def test_gather_threads_follow_affinity_world_and_cpu_quota(monkeypatch):
    """Staging threads per rank: the process's CPUs split between the ranks of the node, never more than the rank's share
    of a container CPU quota (cgroup), 8 at most, the env override wins."""
    import os
    from mvector.predict import MVectorPredictor as P
    monkeypatch.delenv('VPB_GATHER_THREADS', raising=False)
    monkeypatch.setattr(os, 'sched_getaffinity', lambda pid: set(range(128)), raising=False)
    monkeypatch.setattr(os, 'cpu_count', lambda: 128)
    for quota, world, want in ((None, 1, 8), (None, 8, 8), (16.0, 1, 8), (16.0, 8, 2), (16.0, 4, 4), (4.0, 8, 1), (None, 64, 2)):
        monkeypatch.setattr(P, '_quota_cache', [quota])
        monkeypatch.setenv('LOCAL_WORLD_SIZE', str(world))
        assert P._gather_threads() == want, (quota, world)
    # a rank already bound to its own slice (bind_rank_to_local_cpus): the slice is not divided again, the quota still is
    monkeypatch.setattr(os, 'sched_getaffinity', lambda pid: set(range(16)), raising=False)
    monkeypatch.setattr(P, '_quota_cache', [None])
    monkeypatch.setenv('LOCAL_WORLD_SIZE', '8')
    assert P._gather_threads() == 8
    monkeypatch.setattr(P, '_quota_cache', [16.0])
    assert P._gather_threads() == 2
    monkeypatch.setenv('VPB_GATHER_THREADS', '5')
    assert P._gather_threads() == 5


def test_metrics_match_reference_golden():
    """mvector.metric.metrics (metrics.py:5-39) against outputs of the reference's own functions on seeded scores with
    ties (tests/golden/metrics.npz): fnr / fpr / thresholds bit-exact, EER / threshold / minDCF to 1e-12."""
    from mvector.metric.metrics import compute_dcf, compute_eer, compute_fnr_fpr
    z = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'metrics.npz'))
    fnr, fpr, th = compute_fnr_fpr(z['scores'], z['labels'])
    assert np.array_equal(fnr, z['fnr']) and np.array_equal(fpr, z['fpr']) and np.array_equal(th, z['thresholds'])
    eer, thr = compute_eer(fnr, fpr, z['scores'])
    assert abs(eer - float(z['eer'])) < 1e-12 and float(thr) == float(z['threshold'])
    assert abs(compute_eer(fnr, fpr) - float(z['eer'])) < 1e-12
    assert abs(compute_dcf(fnr, fpr) - float(z['min_dcf'])) < 1e-12
    assert abs(compute_dcf(fnr, fpr, p_target=0.05, c_miss=10, c_fa=1) - float(z['min_dcf_05'])) < 1e-12


def test_evaluate_scoring_matches_reference_golden():
    """The score list the reference's evaluate built (trainer.py:452-468, captured by make_golden.py) -> same EER /
    minDCF / threshold through the mirror's metric functions."""
    from mvector.metric.metrics import compute_dcf, compute_eer, compute_fnr_fpr
    z = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'evaluate_small.npz'))
    fnr, fpr, _ = compute_fnr_fpr(z['scores'], z['labels'])
    eer, thr = compute_eer(fnr, fpr, z['scores'])
    assert abs(float(eer) - float(z['eer'])) < 1e-12 and float(thr) == float(np.float32(z['threshold']))
    assert abs(float(compute_dcf(fnr, fpr)) - float(z['min_dcf'])) < 1e-12


def test_evaluate_host_logic_with_oracle_backend(tmp_path, manifest):
    """evaluate's list handling (duration sort, single-utterance featurize, eval crop, feature-level padding per batch,
    trial-major scoring) checked on CPU: the device pieces (featurizer, backbone) are swapped for the oracle, the
    result must reproduce what the reference's evaluate produced (tests/golden/evaluate_small.npz)."""
    import mvector.trainer as mt
    from oracle import frontend as ofe, models as om
    from mvector.utils.utils import dict_to_object
    m = manifest['evaluate_small']
    z = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'evaluate_small.npz'))
    lists = {}
    for nm, count in (('enroll', m['n_enroll']), ('trials', m['n_trials'])):
        lines = []
        for i in range(count):
            p = tmp_path / f'{nm}_{i}.wav'
            with wave.open(str(p), 'wb') as w:
                w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000)
                w.writeframes(z[f'{nm}_pcm{i}'].astype('<i2').tobytes())
            lines.append(f'{p}\t{int(z[f"{nm}_label{i}"])}\n')
        (tmp_path / f'{nm}_list.txt').write_text(''.join(lines))
        lists[nm] = str(tmp_path / f'{nm}_list.txt')
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith('sd/')}
    fargs = dict(m['preprocess']['method_args'])

    class Fz:
        def __call__(self, w):
            return ofe.featurize(w.numpy(), None, 'Fbank', fargs)

        def num_frames(self, n):
            return 1 + (n - 400) // 160

    class Net:
        def eval(self):
            return self

        def __call__(self, x):
            return om.forward(m['model'], sd, x, **m['model_args'])

    tr = object.__new__(mt.MVectorTrainer)
    tr.configs = dict_to_object({'dataset_conf': {'dataset': {'sample_rate': 16000, 'use_dB_normalization': True,
                                                              'target_dB': -20},
                                                  'eval_conf': dict(m['eval_conf']), 'enroll_list': lists['enroll'],
                                                  'trials_list': lists['trials']}})
    tr.use_gpu, tr.stop_eval, tr._device = False, False, torch.device('cpu')
    tr.audio_featurizer, tr.model = Fz(), Net()

    # the two device steps of the glue (memset + D2D padding, vp_cosine_scores) get numpy stand-ins here; the real ones are
    # covered on hardware by tests/test_gpu_parity.py::test_evaluate_matches_reference_golden
    def pad(items):
        x = torch.zeros(len(items), max(f.shape[0] for f in items), items[0].shape[1])
        for i, f in enumerate(items):
            x[i, :f.shape[0]] = f
        return x

    def score(t, e):
        tn = t / np.linalg.norm(t, axis=1, keepdims=True)
        en = e / np.linalg.norm(e, axis=1, keepdims=True)
        return (tn @ en.T).astype(np.float32)

    tr._zero_pad_features, tr._cosine_scores = pad, score
    captured = {}
    real = mt.compute_fnr_fpr

    def spy(scores, labels, weights=None):
        captured['scores'], captured['labels'] = scores.copy(), labels.copy()
        return real(scores, labels, weights)

    mt.compute_fnr_fpr = spy
    try:
        eer, min_dcf, thr = tr.evaluate()
    finally:
        mt.compute_fnr_fpr = real
    assert np.array_equal(captured['labels'], z['labels'])
    assert np.abs(captured['scores'] - z['scores']).max() < 2e-6
    assert abs(eer - float(z['eer'])) < 1e-9 and abs(min_dcf - float(z['min_dcf'])) < 1e-9


def test_diarization_glue_matches_reference_golden():
    """SURVEY.md 8(f) row 4: infer_utils.speaker_diarization (chunking, spectral clustering, cosine merge, post-processing)
    against outputs of the reference's own classes on seeded inputs (tests/golden/diarization.npz)."""
    from mvector.infer_utils.speaker_diarization import SpeakerDiarization, SpectralCluster
    z = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'diarization.npz'))
    sd = SpeakerDiarization()
    vad = diarization_vad(np.random.RandomState(3))
    assert [[s[0], s[1]] for s in vad] == [z[f'vad{i}_t'].tolist() for i in range(int(z['n_vad']))]
    assert arrays_sha256((str(i), s[2]) for i, s in enumerate(vad)) == str(z['vad_x_sha256'])
    sd._check_audio_list(vad)
    chunks = sd._chunk(vad)
    assert np.array_equal(np.array([[c[0], c[1]] for c in chunks]), z['chunk_times'])
    assert np.allclose([float(np.abs(c[2]).sum()) for c in chunks], z['chunk_sums'], rtol=0, atol=0)
    assert all(c[2].shape[0] == 24000 for c in chunks)
    for tag, k in (('auto', None), ('k2', 2), ('k3', 3)):
        np.random.seed(0)
        labels, centres = sd.clustering(z['emb'].copy(), speaker_num=k)
        assert np.array_equal(labels, z[f'labels_{tag}']), tag
        assert np.allclose(centres, z[f'centres_{tag}'], atol=1e-6)
        out = sd.postprocess([list(c) for c in chunks], labels)
        got = np.array([[o['speaker'], o['start'], o['end']] for o in out], dtype=np.float64)
        assert np.array_equal(got, z[f'out_{tag}']), tag
    # pieces
    sc = SpectralCluster()
    A = sc.get_sim_mat(z['emb'])
    assert np.allclose(np.diag(A), 1, atol=1e-6) and np.allclose(A, A.T, atol=1e-6)
    P = sc.p_pruning(A.copy())
    assert ((P != 0).sum(axis=1) == A.shape[0] - int((1 - 6.0 / A.shape[0]) * A.shape[0])).all()
    assert SpeakerDiarization._correct_labels(np.array([2, 2, 0, 1, 0])).tolist() == [0, 0, 1, 2, 1]


def test_energy_vad_and_diarization_segments():
    from mvector.audio import AudioSegment
    from mvector.infer_utils.speaker_diarization import SpeakerDiarization
    rng = np.random.RandomState(0)
    x = np.concatenate([np.zeros(8000), 0.2 * rng.randn(48000), np.zeros(16000), 0.1 * rng.randn(64000),
                        np.zeros(4000)]).astype(np.float32)
    seg = AudioSegment(x, 16000)
    v = seg.vad(return_seconds=True)
    assert len(v) == 2 and abs(v[0]['start'] - 0.5) < 0.05 and abs(v[0]['end'] - 3.5) < 0.05
    assert abs(v[1]['start'] - 4.5) < 0.05 and abs(v[1]['end'] - 8.5) < 0.05
    vs = seg.vad()
    assert vs[0]['start'] == int(round(v[0]['start'] * 16000))
    chunks = SpeakerDiarization().segments_audio(seg)
    assert all(c[2].shape[0] == 24000 for c in chunks) and len(chunks) >= 6
    with pytest.raises(AssertionError):                       # < 5 s of speech: the reference refuses too
        SpeakerDiarization().segments_audio(AudioSegment(x[:40000], 16000))


def _header_struct_fields(name):
    """Field names of ``typedef struct <name> { ... } <name>;`` in include/vpb200.h, in declaration order."""
    src = open(os.path.join(os.path.dirname(__file__), '..', 'include', 'vpb200.h')).read()
    body = re.search(r'typedef struct %s \{(.*?)\} %s;' % (name, name), src, re.S).group(1)
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    fields = []
    for decl in body.split(';'):
        decl = decl.strip()
        if not decl:
            continue
        ctype, names = decl.split(None, 1)
        for n in names.split(','):
            n = n.strip()
            m = re.match(r'(\w+)\[(\d+)\]', n)
            fields.append((ctype, m.group(1), int(m.group(2))) if m else (ctype, n, 1))
    return fields


def test_ctypes_structs_follow_the_header_field_by_field():
    """vp_op / vp_frontend_desc in mvector/_lib.py must list exactly the header's fields, in order, with matching types
    (the sizeof self-check at load time cannot see two swapped int32 fields)."""
    from mvector import _lib
    ctype_of = {'int32_t': ctypes.c_int32, 'int64_t': ctypes.c_int64, 'float': ctypes.c_float}
    for cname, cls in (('vp_op', _lib.Op), ('vp_frontend_desc', _lib.FrontendDesc)):
        want = _header_struct_fields(cname)
        got = list(cls._fields_)
        assert len(want) == len(got), cname
        for (ctype, name, count), (pname, ptype) in zip(want, got):
            assert name == pname, (cname, name, pname)
            assert ptype == (ctype_of[ctype] * count if count > 1 else ctype_of[ctype]), (cname, name)


def test_golden_fixtures_are_complete_and_small(manifest):
    gdir = os.path.join(os.path.dirname(__file__), 'golden')
    total = 0
    for name in manifest:
        if name.startswith('_'):
            continue
        path = os.path.join(gdir, name + '.npz')
        assert os.path.exists(path), f'{name}.npz is listed in manifest.json but missing'
        total += os.path.getsize(path)
    assert total < 24 << 20, 'golden fixtures are meant to stay small (they travel with every gpurun snapshot)'


def test_pack_tc16_image_roundtrip():
    """Experimental fp16 split weight image (engine.pack_tc16): hi + lo reproduces W * 2^k to ~2^-22, the layout decodes
    back through the swizzle, padding rows / columns are zero, descale = 2^-k."""
    from mvector.engine import pack_tc16, tc_tile_n, unpack_tc16
    rng = np.random.default_rng(3)
    for N, K in ((512, 512), (1536, 1536), (192, 200), (128, 72)):
        W = rng.standard_normal((N, K)) * 0.05
        bn = tc_tile_n(N, K > 1536)
        img, descale = pack_tc16(W, bn)
        nt, kb = (N + bn - 1) // bn, (K + 63) // 64
        assert img.dtype == np.float32 and img.size * 4 == nt * kb * 2 * bn * 128
        k = -int(round(np.log2(descale)))
        assert descale == 2.0 ** -k and 2.0 ** 13 < np.abs(W).max() * 2.0 ** k <= 2.0 ** 14
        hi, lo = unpack_tc16(img, N, K, bn)
        err = np.abs((hi.astype(np.float64) + lo) * descale - W).max() / np.abs(W).max()
        assert err < 2.0 ** -21, err
        assert np.abs(lo).max() <= np.abs(hi).max() * 2.0 ** -10


def test_program_export_roundtrip_and_c_host_builds(tmp_path):
    """tools/export_program.py writes (ops, weights) for a C host; examples/embed_from_c.c is a pure-C client of
    include/vpb200.h: the file round-trips, the example compiles as C against the header, and without a GPU it fails
    loudly (no CPU path)."""
    import shutil
    import subprocess
    root = os.path.join(os.path.dirname(__file__), '..')
    sys_path_added = root not in __import__('sys').path
    if sys_path_added:
        __import__('sys').path.insert(0, root)
    from tools import export_program as ex
    from mvector.models import build_model
    from mvector.utils.utils import dict_to_object
    from oracle import models as om
    margs = dict(embd_dim=32, channels=64)
    model = build_model(80, dict_to_object({'model_conf': {'model': 'TDNN', 'model_args': margs}}))
    model.load_state_dict({'0.' + k: v for k, v in om.random_state_dict('TDNN', 80, seed=1, **margs).items()})
    path = str(tmp_path / 'tdnn.vpb')
    pb, blob = ex.export(model, 3, 90, path)
    back = ex.load(path)
    assert (back['B'], back['T'], back['F'], back['embd_dim']) == (3, 90, 80, 32)
    assert back['input_floats'] == 3 * 90 * 80 and back['output_floats'] == 3 * 32
    assert np.array_equal(back['weights'], blob)
    assert len(back['ops']) == len(pb.ops) and all(bytes(a) == bytes(b) for a, b in zip(back['ops'], pb.ops))
    if shutil.which('gcc') is None or not os.path.exists('/usr/local/cuda/include/cuda_runtime_api.h'):
        pytest.skip('no C toolchain / CUDA headers here')
    import __graft_entry__ as ge
    libdir = os.path.dirname(os.path.abspath(ge.build()))           # builds libvpb200.so when it is missing / stale
    exe = str(tmp_path / 'embed_from_c')
    r = subprocess.run(['gcc', '-O1', '-Wall', '-Werror', '-I', os.path.join(root, 'include'), '-I', '/usr/local/cuda/include',
                        os.path.join(root, 'examples', 'embed_from_c.c'), '-o', exe, '-L', libdir, '-lvpb200',
                        '-L', '/usr/local/cuda/lib64', '-lcudart', '-lm', '-Wl,-rpath,' + libdir],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    if not torch.cuda.is_available():
        r = subprocess.run([exe, path], capture_output=True, text=True)
        assert r.returncode == 3 and 'no CPU path' in r.stderr
