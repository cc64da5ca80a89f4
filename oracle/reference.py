"""Install the UNMODIFIED reference (yeyupiaoling/VoiceprintRecognition-Pytorch, mvector 1.1.1) into ``oracle/_ref/``
for bench.py's reference arm (baseline/ref_driver.py) and tests/test_bench_cpu.py.

The reference is pure Python, so installing it is what ``pip install --no-deps --target`` would do: the files of its
``mvector`` package copied as is.  The checkout is taken from ``$VPB_REFERENCE`` or, by default, ``/root/reference``.
Without a readable checkout nothing is installed and the reference arm reports itself unavailable.  ``oracle/_ref/`` is
git-ignored and, once installed, is left as it is (the tree may be read-only where the benchmark runs)."""
import os
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, '_ref')


def installed():
    return os.path.isfile(os.path.join(DEST, 'mvector', '__init__.py'))


def install(source=None):
    """Copy ``<source>/mvector`` to ``oracle/_ref/mvector`` unless it is there already.  Returns DEST when the reference
    is installed, None when no readable checkout exists or the install fails (said on stderr)."""
    if installed():
        return DEST
    source = source or os.environ.get('VPB_REFERENCE', '/root/reference')
    pkg = os.path.join(source, 'mvector')
    if not os.access(os.path.join(pkg, '__init__.py'), os.R_OK):
        return None
    tmp = None
    try:                                   # copied aside first: a partial copy never looks installed
        os.makedirs(DEST, exist_ok=True)
        tmp = tempfile.mkdtemp(dir=DEST)
        for root, dirs, files in os.walk(pkg):
            dirs[:] = [d for d in dirs if d != '__pycache__']
            out = os.path.join(tmp, 'mvector', os.path.relpath(root, pkg))
            os.makedirs(out)               # contents only, not modes: a read-only checkout still gives a tree the
            for f in files:                # installing user can move into place and later delete
                if not f.endswith('.pyc'):
                    shutil.copyfile(os.path.join(root, f), os.path.join(out, f))
        os.rename(os.path.join(tmp, 'mvector'), os.path.join(DEST, 'mvector'))
    except OSError as e:
        sys.stderr.write(f'oracle.reference: reference at {source} not installed into {DEST}: {e}\n')
        return None
    finally:
        if tmp:
            shutil.rmtree(tmp, ignore_errors=True)
    return DEST
