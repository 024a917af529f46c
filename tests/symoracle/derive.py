"""TEST-ONLY loader of tests/symoracle/derive_oracle.c: the C oracle's Keypair::derive over a batch on all host cores.  The library is
built with gcc into the temporary directory, so the repository tree stays unchanged."""
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
        src = os.path.join(_HERE, "derive_oracle.c")
        deps = [src] + [os.path.join(_ROOT, "oracle", "c", f) for f in ("afx_oracle.c", "prim.h", "consts.h")]
        so = os.path.join(tempfile.gettempdir(), "afx_derive_oracle_%d.so" % os.getuid())
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            tmp = so + ".%d" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-pthread", "-fvisibility=hidden", "-o", tmp, src])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        L.afxd_derive.restype = ctypes.c_double
        L.afxd_derive.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int,
                                  ctypes.c_void_p]
        _lib = L
    return _lib


def derive(sysparams, issuer_pub, master_secrets, threads=0):
    """master secrets [count][64] -> (keypairs [count][128] = a || a0 || a1 || pk under sysparams, seconds)"""
    ms = np.ascontiguousarray(master_secrets, dtype=np.uint8)
    out = np.zeros((ms.shape[0], 128), np.uint8)
    secs = lib().afxd_derive(sysparams, len(sysparams), issuer_pub, ms.ctypes.data, ms.shape[0], threads or os.cpu_count(), out.ctypes.data)
    if secs < 0:
        raise ValueError("system parameters or issuer key do not parse")
    return out, secs
