"""Helpers shared by the tests and tests/golden/make_golden.py for fixture data regenerated from seeds instead of stored
(plain module: generating fixtures needs no pytest)."""
import hashlib

import numpy as np


def arrays_sha256(named_arrays):
    """SHA-256 over (name, dtype, shape, bytes) of every array in order: pins a seeded fixture input that is regenerated
    instead of stored, and a reference output too large to store whole."""
    h = hashlib.sha256()
    for k, v in named_arrays:
        v = np.ascontiguousarray(np.asarray(v))
        h.update(f'{k}:{v.dtype.str}:{v.shape};'.encode())
        h.update(v.tobytes())
    return h.hexdigest()


def diarization_vad(rng, sr=16000):
    """The synthetic VAD segments ``[start s, end s, samples]`` of tests/golden/diarization.npz drawn from ``rng``: 4.1,
    0.9, 6.35, 2.0 and 3.77 s of noise 0.4 s apart, each cut or padded to int(end * sr) - int(start * sr) samples."""
    segs, t0 = [], 0.0
    for dur in (4.1, 0.9, 6.35, 2.0, 3.77):
        n = int((t0 + dur) * sr) - int(t0 * sr)
        segs.append([round(t0, 3), round(t0 + dur, 3), rng.randn(n).astype(np.float32)])
        t0 = round(t0 + dur + 0.4, 3)
    for seg in segs:
        want = int(seg[1] * sr) - int(seg[0] * sr)
        seg[2] = seg[2][:want]
        if seg[2].shape[0] < want:
            seg[2] = np.pad(seg[2], (0, want - seg[2].shape[0]))
    return segs
