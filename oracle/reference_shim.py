"""Loader that imports the UNMODIFIED reference (python-2 code) under python 3.

TEST INFRASTRUCTURE.  Sources come from /root/reference where it is mounted (the build container)
or from the byte-identical staged copy oracle/_ref/ (``oracle/make_ref.py``; git-ignored).  Used by
``oracle/make_golden.py`` to freeze fixtures and by ``oracle/cpu_bench.py`` to time the reference's
own code.  Recipe: SURVEY.md appendix C.
"""
import os
import pickle
import sys
import tempfile
import types

REFERENCE_ROOT = "/root/reference"
STAGED_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


class Py2Int(int):
    """``fft_n/2`` must stay an int (mfcc.py:45,46,61 rely on python-2 division)."""

    def __truediv__(self, o):
        return Py2Int(int.__floordiv__(self, o)) if isinstance(o, int) else float(self) / o


def root():
    """Directory the reference modules are imported from, or None."""
    if os.path.isfile(os.path.join(REFERENCE_ROOT, "mfcc.py")):
        return REFERENCE_ROOT
    from . import make_ref
    return STAGED_ROOT if make_ref.staged_ok() else None


def available():
    return root() is not None


_cache = {}


def load():
    """Returns a namespace with the reference modules ``mfcc``, ``file_processing``,
    ``sklearn_analyser`` and the python-2-int ``FFT_N``."""
    if "ns" in _cache:
        return _cache["ns"]
    base = root()
    if base is None:
        raise RuntimeError("reference neither mounted at %s nor staged under oracle/_ref" % REFERENCE_ROOT)
    for p in (os.path.join(base, "dataset"), os.path.join(base, "realtime_analysis"), base):
        if p not in sys.path:
            sys.path.insert(0, p)
    sys.modules.setdefault("cPickle", pickle)                 # sklearn_analyser.py:1
    sys.modules.setdefault("h5py", types.ModuleType("h5py"))  # dataset/file_index.py:1
    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp(prefix="vadref_"))              # sklearn_analyser.py:10 opens ./analyser.log
    try:
        import mfcc as ref_mfcc
        import file_processing as ref_fp
        import sklearn_analyser as ref_an
    finally:
        os.chdir(cwd)
    ns = types.SimpleNamespace(mfcc=ref_mfcc, file_processing=ref_fp, sklearn_analyser=ref_an,
                               FFT_N=Py2Int(512), root=base)
    _cache["ns"] = ns
    return ns
