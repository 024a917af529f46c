"""TEST-ONLY loader of tests/symoracle/sym_oracle.c: the C oracle's Plaintext::from, Keypair::encrypt and Keypair::decrypt over a
batch on all host cores.  The library is built with gcc into the temporary directory, so the repository tree stays unchanged."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "sym_oracle.c")
        deps = [src] + [os.path.join(_ROOT, "oracle", "c", f) for f in ("afx_oracle.c", "prim.h", "consts.h")]
        so = os.path.join(tempfile.gettempdir(), "afx_sym_oracle_%d.so" % os.getuid())
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            tmp = so + ".%d" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-pthread", "-fvisibility=hidden", "-o", tmp, src])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        vp = ctypes.c_void_p
        L.afxs_run.restype = ctypes.c_double
        L.afxs_run.argtypes = [ctypes.c_int, vp, vp, ctypes.c_uint64, ctypes.c_int, vp, vp, vp]
        _lib = L
    return _lib


def _run(op, keypair, inp, out_shape, with_pt=False, threads=0):
    inp = np.ascontiguousarray(inp, dtype=np.uint8)
    count = inp.shape[0]
    out = np.zeros((count,) + out_shape, np.uint8)
    pt = np.zeros((count, 3, 32), np.uint8) if with_pt else None
    status = np.zeros(count, np.uint8)
    kp = ctypes.create_string_buffer(bytes(keypair)[:96], 96) if keypair is not None else None
    secs = lib().afxs_run(op, ctypes.addressof(kp) if kp is not None else None, inp.ctypes.data, count, threads or os.cpu_count(),
                          out.ctypes.data, pt.ctypes.data if with_pt else None, status.ctypes.data)
    return out, pt, status, secs


def encode(data, threads=0):
    """data [count][30] -> (plaintexts [count][3][32], seconds)"""
    out, _, _, secs = _run(0, None, data, (3, 32), threads=threads)
    return out, secs


def encrypt(keypair, plaintexts, threads=0):
    """-> (ciphertexts [count][2][32], status, seconds)"""
    out, _, status, secs = _run(1, keypair, plaintexts, (2, 32), threads=threads)
    return out, status, secs


def decrypt(keypair, ciphertexts, threads=0):
    """-> (data [count][30], plaintexts [count][3][32], status, seconds)"""
    return _run(2, keypair, ciphertexts, (30,), with_pt=True, threads=threads)
