"""Builds and binds tests/oracle_weighted.c: the CPU oracle's update with importance weights (prioritized replay).  The library is
compiled with the oracle's own flags (oracle/Makefile) into a directory the caller gives (the tree may be read-only), and its function
runs on the handles of oracle.OracleDdpg: both libraries compile the same oracle source, so they share the handle's layout."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
CFLAGS = ["-O3", "-fPIC", "-std=gnu11", "-ffp-contract=off", "-fno-fast-math", "-fexcess-precision=standard", "-fopenmp"]


def load(out_dir):
    so = os.path.join(out_dir, "liboracle_weighted.so")
    subprocess.check_call(["gcc"] + CFLAGS + ["-shared", "-o", so, os.path.join(HERE, "oracle_weighted.c"),
                                             os.path.join(ORACLE, "shems_oracle.c"), "-lm"])
    L = C.CDLL(so)
    PF = C.POINTER(C.c_float)
    L.oracle_ddpg_update_batch_weighted.argtypes = [C.c_void_p, PF, PF, PF, PF, PF, PF, PF, PF]
    L.oracle_ddpg_update_batch_weighted.restype = None
    return L


def update_batch_weighted(L, orc, s, a, r, s2, done, w):
    """orc (oracle.OracleDdpg).update_batch with the critic's dq of row b scaled by w[b]; returns (q, y) of the critic step"""
    f = lambda x: np.ascontiguousarray(x, np.float32)
    fp = lambda x: x.ctypes.data_as(C.POINTER(C.c_float)) if x is not None else None
    B = np.asarray(r).size
    q, y = np.zeros(B, np.float32), np.zeros(B, np.float32)
    arrs = [f(s), f(a), f(r), f(s2), f(done) if done is not None else None, f(w)]
    L.oracle_ddpg_update_batch_weighted(C.c_void_p(orc.h), *[fp(x) for x in arrs], fp(q), fp(y))
    return q, y
