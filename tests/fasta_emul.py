"""TEST INFRASTRUCTURE: the contigs FASTA reading's stage functions
(gt-scaffold_b200/csrc/gtsb_fasta_core.h, the bodies of the kp_fa_* kernels in gtsb_parse.cu)
compiled for the host and run as plain loops (tests/emul/fasta_emul.cpp).  Used by
tests/test_fasta.py and tests/test_fasta_gpu.py to check the device against the same stages
without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "gt-scaffold_b200", "csrc")
SRC = os.path.join(HERE, "emul", "fasta_emul.cpp")
CORES = [os.path.join(CSRC, "gtsb_fasta_core.h"), os.path.join(CSRC, "gtsb_parse_core.h")]
OUT = os.path.join(HERE, "emul", "_build", "libfasta_emul.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(OUT) or os.path.getmtime(OUT) < max(os.path.getmtime(f) for f in [SRC] + CORES):
            os.makedirs(os.path.dirname(OUT), exist_ok=True)
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", OUT, SRC], check=True)
        _lib = C.CDLL(OUT)
        _lib.emul_fasta.restype = C.c_uint32
    return _lib


def read(text, min_len, order):
    """the stage functions as host loops -> (irregular, headers in id order, seq_len by id); order 0
    visits the lines forwards, 1 backwards, 2 in a scrambled order"""
    L = lib()
    n = len(text)
    V = C.c_uint64(0)
    buf = np.zeros(n + 8, np.uint8)
    buf[:n] = np.frombuffer(text, np.uint8)
    names = np.zeros(n + 1, np.uint8)
    off = np.zeros(n + 2, np.uint64)
    seq = np.zeros(n + 1, np.uint64)
    irr = L.emul_fasta(buf.ctypes.data_as(C.c_void_p), C.c_uint64(n), C.c_uint64(min_len), C.c_int(order),
                       names.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p),
                       seq.ctypes.data_as(C.c_void_p), C.byref(V))
    if irr:
        return irr, None, None
    raw, o = names.tobytes(), off.tolist()
    return 0, [raw[o[i]:o[i + 1]] for i in range(V.value)], seq[:V.value].tolist()
