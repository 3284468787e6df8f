"""ctypes wrapper around oracle/libmyo_oracle.so (CPU oracle; test infrastructure only)."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "libmyo_oracle.so")
    deps = [os.path.join(_HERE, "myo_oracle.c"), os.path.join(_HERE, "..", "include", "myo_blob_layout.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-B"])
    return so


def build_native():
    """-O3 -march=native build for the timed CPU arm (bench.py --impl reference), compiled ON the machine that runs it into a temporary
    directory removed at exit, so that benchmarking writes nothing into the tree.  Falls back to the portable build if the compiler refuses."""
    d = tempfile.mkdtemp(prefix="myo_oracle_native_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "libmyo_oracle_native.so")
    try:
        subprocess.check_call(["gcc", "-O3", "-march=native", "-fPIC", "-std=c11", "-ffp-contract=off", "-shared", "-o", so, os.path.join(_HERE, "myo_oracle.c"), "-lm"],
                              stderr=subprocess.DEVNULL)
        return so
    except Exception:
        return build()


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(os.environ.get("MYO_ORACLE_LIB") or build())
        L.oracle_create.restype = ctypes.c_void_p
        L.oracle_create.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.oracle_field.restype = ctypes.POINTER(ctypes.c_double)
        L.oracle_field.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_int)]
        L.oracle_ifield.restype = ctypes.POINTER(ctypes.c_int)
        L.oracle_ifield.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_int)]
        for f in ("oracle_forward", "oracle_step", "oracle_reset", "oracle_destroy"):
            getattr(L, f).argtypes = [ctypes.c_void_p]
            getattr(L, f).restype = None
        L.oracle_step_n.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.oracle_step_n.restype = None
        L.oracle_info.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.oracle_info.restype = ctypes.c_int
        _LIB = L
    return _LIB


class Oracle:
    """One env of the CPU oracle.  `I`, `D` are the packed model blob (myosuite_b200.blob.pack)."""

    def __init__(self, I, D):
        self._I = np.ascontiguousarray(I, dtype=np.int32)
        self._D = np.ascontiguousarray(D, dtype=np.float64)
        self._L = lib()
        self._h = self._L.oracle_create(self._I.ctypes.data, self._D.ctypes.data)
        if not self._h:
            raise RuntimeError("oracle_create failed (blob magic/version)")

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.oracle_destroy(self._h)
            self._h = None

    def f(self, name):
        """numpy VIEW of a float64 field (valid until the next forward/step for variable-size ones)."""
        n = ctypes.c_int(0)
        p = self._L.oracle_field(self._h, name.encode(), ctypes.byref(n))
        if not p:
            raise KeyError(name)
        return np.ctypeslib.as_array(p, shape=(max(n.value, 0),)) if n.value else np.zeros(0)

    def i(self, name):
        n = ctypes.c_int(0)
        p = self._L.oracle_ifield(self._h, name.encode(), ctypes.byref(n))
        return np.ctypeslib.as_array(p, shape=(n.value,)).copy() if n.value else np.zeros(0, np.int32)

    def set(self, **kw):
        for k, v in kw.items():
            self.f(k)[:] = v

    def reset(self):
        self._L.oracle_reset(self._h)

    def forward(self):
        self._L.oracle_forward(self._h)

    def step(self, n=1):
        self._L.oracle_step_n(self._h, n)

    @property
    def ncon(self):
        return self._L.oracle_info(self._h, 0)

    @property
    def nefc(self):
        return self._L.oracle_info(self._h, 1)

    @property
    def solver_niter(self):
        return self._L.oracle_info(self._h, 4)
