"""ctypes wrapper over tools/corpus_gen.c (synthetic corpora of SURVEY.md §8(d)).  Test/bench infrastructure."""
import ctypes, os, subprocess, tempfile
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libcorpus.so")
_SRC = os.path.join(_HERE, "corpus_gen.c")


def build(force=False):
    """Path of the generator library, compiled when missing or older than its source (into a temporary directory when
    the tree is read-only)."""
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        so = _SO if os.access(_HERE, os.W_OK) else os.path.join(tempfile.mkdtemp(prefix="b2t_corpus_"), "libcorpus.so")
        subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-o", so, _SRC, "-lm"])
        return so
    return _SO


_lib = None


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(build())
        lib.b2t_corpus_open.restype = ctypes.c_void_p
        lib.b2t_corpus_open.argtypes = [ctypes.c_int, ctypes.c_uint64]
        lib.b2t_corpus_close.argtypes = [ctypes.c_void_p]
        lib.b2t_corpus_generate.restype = ctypes.c_uint64
        lib.b2t_corpus_generate.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p,
                                            ctypes.c_uint64, ctypes.c_void_p]
        _lib = lib
    return _lib


def generate(kind, seed, first_doc, n_docs, max_bytes=None, out=None):
    """Return (bytes: np.uint8[total], doc_off: np.uint64[n+1]) for docs [first_doc, first_doc+n_docs).

    If max_bytes is given, generation stops at the first doc that might overflow it (fewer docs returned).
    `out` may be a pre-allocated (e.g. pinned) uint8 array to generate into.
    """
    lib = _load()
    if out is None:
        cap = int(max_bytes) + 200000 if max_bytes is not None else int(n_docs) * 9000 + 200000
        if kind == 5:
            cap = int(max_bytes) + 200000 if max_bytes is not None else int(n_docs) * 140000 + 200000
        out = np.empty(cap, dtype=np.uint8)
    cap = out.size if max_bytes is None else min(out.size, int(max_bytes) + 140000)
    doc_off = np.empty(int(n_docs) + 1, dtype=np.uint64)
    h = lib.b2t_corpus_open(kind, seed)
    try:
        n = lib.b2t_corpus_generate(h, first_doc, n_docs, out.ctypes.data, cap, doc_off.ctypes.data)
    finally:
        lib.b2t_corpus_close(h)
    doc_off = doc_off[: n + 1]
    return out[: int(doc_off[-1])], doc_off


def to_strings(data, doc_off):
    b = data.tobytes()
    return [b[int(doc_off[i]): int(doc_off[i + 1])].decode("utf-8") for i in range(len(doc_off) - 1)]
