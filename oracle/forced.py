"""Forced playouts at the root (Wu 2019, section 3.2) for the CPU oracle.
TEST INFRASTRUCTURE ONLY.

ctypes wrapper over ``oracle/build/libazalea_oracle_forced.so``, built from
forced.c and linked against the oracle's own library: the functions here work
on ``oracle.Tree`` / ``oracle.Hex`` objects.  With ``forced_k = 0`` they are
the oracle's ``select_batch`` / ``sample_paths_stub``, bit for bit.
"""
import ctypes as C
import os
import subprocess

from . import OHex, OLeaves, OTree, SearchTreeFull
from . import build as build_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, 'build', 'libazalea_oracle_forced.so')
# the oracle's own flags (Makefile): float32 arithmetic never fuses a*b+c
_CFLAGS = ['-O2', '-fPIC', '-ffp-contract=off', '-fno-fast-math', '-Wall', '-Wextra', '-std=gnu11']


def build(force=False):
    """Compile forced.c against the oracle's library with gcc (idempotent)."""
    base = build_oracle()
    src = os.path.join(_HERE, 'forced.c')
    hdr = os.path.join(_HERE, 'azalea_oracle.h')
    if (not force and os.path.exists(_LIB_PATH)
            and os.path.getmtime(_LIB_PATH) >= max(os.path.getmtime(src), os.path.getmtime(hdr),
                                                   os.path.getmtime(base))):
        return _LIB_PATH
    subprocess.check_call([os.environ.get('CC', 'gcc')] + _CFLAGS + [
        '-shared', '-o', _LIB_PATH, src, '-L' + os.path.dirname(base), '-lazalea_oracle',
        '-Wl,-rpath,$ORIGIN', '-lm'], cwd=_HERE)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    from . import lib as oracle_lib
    oracle_lib()                # the oracle's library first: this one resolves against it
    build()
    L = C.CDLL(_LIB_PATH)
    L.omcts_select_batch_forced.argtypes = [C.POINTER(OTree), C.POINTER(OHex), C.c_int,
                                            C.c_float, C.c_float, C.POINTER(OLeaves)]
    L.omcts_sample_paths_stub_forced.argtypes = [C.POINTER(OTree), C.POINTER(OHex), C.c_int,
                                                 C.c_int, C.c_float, C.c_float, C.c_int,
                                                 C.POINTER(C.c_float)]
    _lib = L
    return L


def select_batch(tree, game, batch_size, coef, forced_k):
    """``tree.select_batch`` with forced playouts at the root."""
    rc = lib().omcts_select_batch_forced(tree.t, C.byref(game.g), batch_size, C.c_float(coef),
                                         C.c_float(forced_k), C.byref(tree._lv))
    if rc < 0:
        raise AssertionError('oracle select failed: %d' % rc)
    return tree._leaves(game.n)


def sample_paths_stub(tree, game, num_simulations, batch_size, coef, stub_mode, forced_k):
    """``tree.sample_paths_stub`` with forced playouts at the root."""
    sv = C.c_float()
    rc = lib().omcts_sample_paths_stub_forced(tree.t, C.byref(game.g), num_simulations,
                                              batch_size, C.c_float(coef), C.c_float(forced_k),
                                              stub_mode, C.byref(sv))
    if rc == -1:
        raise SearchTreeFull('too many nodes')
    if rc < 0:
        raise AssertionError('oracle search failed: %d' % rc)
    return float(sv.value)
