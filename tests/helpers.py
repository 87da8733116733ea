"""Shared test helpers: oracle / reference / emulation loaders and golden fixtures (TEST ONLY)."""
import ctypes
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
DEFAULT = [3, -6, -5, -2]


def porechop_checkout():
    """A checkout of rrwick/Porechop (its Python package and test fixtures), which the tests that run its CLI need and
    skip without: $PORECHOP_CHECKOUT, else the checkout oracle/_ref was built from (oracle/Makefile `ref`), else ''."""
    path = os.environ.get('PORECHOP_CHECKOUT', '')
    if not path:
        try:
            with open(os.path.join(ROOT, 'oracle', '_ref', 'checkout')) as f:
                path = f.read().strip()
        except OSError:
            pass
    return path if path and os.path.isdir(path) else ''


PORECHOP_CHECKOUT = porechop_checkout()


class Rec(ctypes.Structure):
    _fields_ = [('v', ctypes.c_int32 * 9)]


def _abi(lib):
    lib.adapterAlignment.argtypes = [ctypes.c_char_p, ctypes.c_char_p] + [ctypes.c_int] * 4
    lib.adapterAlignment.restype = ctypes.c_void_p
    lib.freeCString.argtypes = [ctypes.c_void_p]
    return lib


_cache = {}


def oracle_lib():
    if 'o' not in _cache:
        lib = _abi(ctypes.CDLL(os.path.join(ROOT, 'oracle', 'liboracle.so')))
        lib.oracle_align_record.argtypes = [ctypes.c_char_p, ctypes.c_int64, ctypes.c_char_p, ctypes.c_int64] + \
            [ctypes.c_int] * 4 + [ctypes.POINTER(Rec)]
        lib.oracle_align_batch.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64] + \
            [ctypes.c_int] * 4 + [ctypes.c_void_p]
        _cache['o'] = lib
    return _cache['o']


def ref_lib():
    """The unmodified reference C++ (oracle/_ref/cpp_functions.so) or None if it was never built."""
    if 'r' not in _cache:
        p = os.path.join(ROOT, 'oracle', '_ref', 'cpp_functions.so')
        _cache['r'] = _abi(ctypes.CDLL(p)) if os.path.exists(p) else None
    return _cache['r']


def emu_lib():
    if 'e' not in _cache:
        lib = ctypes.CDLL(os.environ.get('PB200_EMU_LIB') or os.path.join(ROOT, 'tests', 'emu', 'libemu.so'))
        lib.emu_align_slot.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int,
                                       ctypes.c_char_p, ctypes.c_int] + [ctypes.c_int] * 9 + [ctypes.POINTER(ctypes.c_int32)] * 2
        _cache['e'] = lib
    return _cache['e']


def abi_string(lib, read, adapter, sc):
    p = lib.adapterAlignment(read.encode(), adapter.encode(), *sc)
    s = ctypes.cast(p, ctypes.c_char_p).value.decode()
    lib.freeCString(p)
    return s


def oracle_string(read, adapter, sc=DEFAULT):
    return abi_string(oracle_lib(), read, adapter, sc)


def oracle_record(read, adapter, sc=DEFAULT):
    r = Rec()
    rb, ab = read.encode(), adapter.encode()
    assert oracle_lib().oracle_align_record(rb, len(rb), ab, len(ab), *sc, ctypes.byref(r)) == 0
    return list(r.v)


def oracle_batch(seq_buf, seq_off, ad_buf, ad_off, sc, pair_seq=None, pair_adapter=None):
    seq_buf = np.ascontiguousarray(seq_buf, dtype=np.uint8)
    seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
    ad_buf = np.ascontiguousarray(ad_buf, dtype=np.uint8)
    ad_off = np.ascontiguousarray(ad_off, dtype=np.int32)
    n_seqs, n_ad = len(seq_off) - 1, len(ad_off) - 1
    n_pairs = n_seqs * n_ad if pair_seq is None else len(pair_seq)
    out = np.empty((n_pairs, 9), dtype=np.int32)
    ps = None if pair_seq is None else np.ascontiguousarray(pair_seq, dtype=np.int32)
    pa = None if pair_adapter is None else np.ascontiguousarray(pair_adapter, dtype=np.int32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p) if a is not None else None
    rc = oracle_lib().oracle_align_batch(p(seq_buf), p(seq_off), n_seqs, p(ad_buf), p(ad_off), n_ad, p(ps), p(pa), n_pairs,
                                         *[int(x) for x in sc], p(out))
    assert rc == 0
    return out


def emu_slot(a, b, G, R, mode, sc):
    """a, b: (read, adapter) or b None.  Returns (status, recA, recB)."""
    ra = (ctypes.c_int32 * 9)()
    rb = (ctypes.c_int32 * 9)()
    mx = max(sc[0], sc[1], 0)
    den = min(abs(sc[2]), abs(sc[3])) or 1
    nb = len(b[0]) if b else -1
    st = emu_lib().emu_align_slot(a[0].encode(), len(a[0]), a[1].encode(), len(a[1]), (b[0] if b else '').encode(), nb,
                                  (b[1] if b else '').encode(), len(b[1]) if b else 0, G, R, mode, *sc, mx, den, ra, rb)
    return st, list(ra), list(rb)


def load_golden(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def class_geometry(m):
    """(G, R) of the trace kernel the engine picks for an adapter of length m (engine.cu class_of):
    the smallest capacity G*R >= m with G in {4,8,16,32}, R in {5,6,7,8}."""
    for k in range(16):
        G, R = 4 << (k // 4), 5 + (k % 4)
        if m <= G * R:
            return G, R
    return 32, 8
