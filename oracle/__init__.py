"""CPU oracle for the waveform -> speaker-embedding path.

TEST INFRASTRUCTURE ONLY.  This package is a CPU (torch fp32 / numpy) restatement of the
reference's algorithm for the hot path.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import it, and only as the
checker (or as the timed CPU baseline) -- never on the product path.  The product package
(``voiceprintrecognition-pytorch_b200``) never imports ``oracle`` and fails loudly when its
CUDA library is missing.  ``oracle.reference`` is the one module ``build()`` uses: it installs the unmodified
reference into ``oracle/_ref/`` for ``bench.py``'s reference arm.

Pinning: the reference ships no tests / golden vectors (SURVEY.md section 4), so the oracle is
pinned against outputs of the reference itself, generated in the authoring container by
``tests/golden/make_golden.py`` (imports /root/reference) and committed under ``tests/golden``.
``tests/test_oracle_golden.py`` re-checks the oracle against those fixtures on every run, and
``tests/test_oracle_vs_reference.py`` against the reference's full-size outputs in ``tests/golden/full_size.npz``.

Reference citations are relative to /root/reference (``kaldi.py`` = torchaudio/compliance/kaldi.py,
``functional.py`` = torchaudio/functional/functional.py of torchaudio 2.11.0).
"""
