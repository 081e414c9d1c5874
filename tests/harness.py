"""What several test modules share: the C++ oracles and mirror programs they build, a fresh process on emulated devices, and the
case builders and oracle wrappers of the SRS and keygen tests."""
import ctypes
import os
import subprocess
import sys
import tempfile

import numpy as np

import bn254 as o
import parity_cases as pc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_LIB = os.path.join(ROOT, "tools", "emu", "libh2b200_emu.so")
R = o.R_MOD
_ORACLES = {}


# ---- building and running ----------------------------------------------------------------------------------------------
def build_oracle(source, argtypes, restypes=None):
    """tests/cpp/<source>.cpp (on oracle/h2_oracle.cpp), built once per process into a temporary directory; sets `argtypes`
    (and `restypes`), {function name: ctypes types}, and returns the library"""
    if source not in _ORACLES:
        so = os.path.join(tempfile.mkdtemp(prefix=source + "_"), "lib%s.so" % source)
        subprocess.check_call(["g++", "-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-Wno-unused-function", "-o", so,
                               os.path.join(ROOT, "tests", "cpp", source + ".cpp")])
        _ORACLES[source] = ctypes.CDLL(so)
    L = _ORACLES[source]
    for name, types in argtypes.items():
        getattr(L, name).argtypes = types
    for name, t in (restypes or {}).items():
        getattr(L, name).restype = t
    return L


def build_mirror(source, lib_path, tmp_path):
    """tests/cpp/<source>.cpp, a C++ program on halo2_scaffold_b200/host/h2b200.hpp, linked against the library at lib_path -> its path"""
    exe = str(tmp_path / source)
    libdir, libfile = os.path.split(lib_path)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-o", exe, os.path.join(ROOT, "tests", "cpp", source + ".cpp"),
                           "-L" + libdir, "-l:" + libfile, "-Wl,-rpath," + libdir])
    return exe


def run_on_emulated_devices(module, body, devices, env=None, timeout=1200):
    """`body` in a fresh process on the emulator build, which reports `devices` devices (None: its default of one), with `env` added to
    the environment (the library reads its knobs once).  The body sees np, oc (the oracle), pc (parity_cases), L (the library on every
    device) and, when `module` is named, that test module as t."""
    code = ("import sys; sys.path[:0]=[%r,%r,%r]\n"
            "import numpy as np, oracle_c as oc, parity_cases as pc\n"
            % (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")))
    if module:
        code += "import %s as t\n" % module
    code += "from halo2_scaffold_b200._lib import Lib\nL=Lib(%r, allow_emulator=True); L.init(0)\n" % EMU_LIB
    if devices is not None:
        code += "assert L.device_count() == %s\n" % devices
    code += body + "\nprint('ok')\n"
    env = dict(os.environ, **(env or {}))
    if devices is not None:
        env["H2B_EMU_DEVICES"] = str(devices)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=timeout)
    assert out.returncode == 0 and "ok" in out.stdout, (out.stdout[-1000:], out.stderr[-3000:])


# ---- words and points --------------------------------------------------------------------------------------------------
def threads():
    return os.cpu_count() or 1


def mont(oc, vals):
    return oc.ints_to_words([o.to_mont(v % R, R) for v in vals])


def W(x):
    from halo2_scaffold_b200.domain import fr_to_words
    return fr_to_words(int(x))


def ints(words):
    """Montgomery words -> canonical integers"""
    import oracle_c
    return [o.from_mont(v, R) for v in oracle_c.words_to_ints(np.ascontiguousarray(words, dtype=np.uint64).reshape(-1, 4))]


def affine_ints(oc, pts):
    v = oc.words_to_ints(np.ascontiguousarray(pts).reshape(-1, 4))
    return [None if v[2 * i] == 0 and v[2 * i + 1] == 0 else (o.from_mont(v[2 * i], o.P_MOD), o.from_mont(v[2 * i + 1], o.P_MOD))
            for i in range(len(v) // 2)]


def affine(oc, jacs):
    return np.stack([pc.affine_of(oc, j) for j in np.asarray(jacs).reshape(-1, 12)])


# ---- the SRS -----------------------------------------------------------------------------------------------------------
def orc_srs_setup(k, s, threads=0):
    """ParamsKZG::setup(k, s) of tests/cpp/srs_setup_oracle.cpp -> (g, g_lagrange)"""
    vp = ctypes.c_void_p
    L = build_oracle("srs_setup_oracle", dict(orc_srs_setup=[ctypes.c_uint32, vp, ctypes.c_int, vp, vp]))
    s = np.ascontiguousarray(s, dtype=np.uint64).reshape(4)
    g, gl = np.empty((1 << k, 8), dtype=np.uint64), np.empty((1 << k, 8), dtype=np.uint64)
    L.orc_srs_setup(k, s.ctypes.data, threads or os.cpu_count() or 1, g.ctypes.data, gl.ctypes.data)
    return g, gl


# ---- keygen ------------------------------------------------------------------------------------------------------------
class Consts:
    """the domain constants of EvaluationDomain::new(5, k) (extended_k = k + 2), as words"""

    def __init__(self, L, k):
        import halo2_scaffold_b200 as h2
        from halo2_scaffold_b200 import keygen as kg
        self.dom = h2.EvaluationDomain(5, k, lib=L)
        d = self.dom
        self.k, self.ek, self.n = k, d.extended_k, 1 << k
        self.delta, self.omega, self.omega_inv = W(kg.FR_DELTA), W(d.omega), W(d.omega_inv)
        self.ifft, self.ext_omega = W(d.ifft_divisor), W(d.extended_omega)
        self.zeta = np.stack([W(1), W(d.g_coset), W(d.g_coset_inv)])

    @classmethod
    def on_host(cls, k):
        """the same constants computed on the host alone (no library, no domain object)"""
        import halo2_scaffold_b200.domain as dm
        from halo2_scaffold_b200 import keygen as kg
        c = cls.__new__(cls)
        n, ek = 1 << k, k + 2
        w = dm.FR_ROOT_OF_UNITY
        for _ in range(ek, dm.FR_S):
            w = w * w % R
        ext_omega = w
        for _ in range(k, ek):
            w = w * w % R
        c.k, c.ek, c.n = k, ek, n
        c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega = W(kg.FR_DELTA), W(w), W(pow(w, -1, R)), W(pow(n, -1, R)), W(ext_omega)
        c.zeta = np.stack([W(1), W(dm.FR_ZETA), W(dm.FR_ZETA * dm.FR_ZETA % R)])
        return c


def random_copies(rng, P, n, count, rows=None):
    """copies between random cells (rows < `rows`), with repeated and reversed (redundant) copies mixed in"""
    rows = rows or n
    cs = [(int(rng.integers(P)), int(rng.integers(rows)), int(rng.integers(P)), int(rng.integers(rows))) for _ in range(count)]
    extra = [cs[int(rng.integers(len(cs)))] for _ in range(count // 4)]
    extra += [(d, e, a, b) for (a, b, d, e) in (cs[int(rng.integers(len(cs)))] for _ in range(count // 4))]
    cs += extra
    rng.shuffle(cs)
    return cs


def orc_mapping(P, k, copies):
    """Assembly's mapping after `copies` of tests/cpp/permutation_keygen_oracle.cpp -> (P, n, 2) (column, row)"""
    vp, u32 = ctypes.c_void_p, ctypes.c_uint32
    L = build_oracle("permutation_keygen_oracle", dict(orc_assembly_mapping=[u32, u32, vp, ctypes.c_size_t, vp]))
    c = np.ascontiguousarray(np.array(copies, dtype=np.uint64).reshape(-1, 4))
    out = np.empty((P, 1 << k, 2), dtype=np.uint64)
    L.orc_assembly_mapping(P, k, c.ctypes.data, c.shape[0], out.ctypes.data)
    return out


def sparse(rng, S, n, density):
    return rng.random((S, n)) < density


def disjoint(S, n, stride=None):
    """selector s active on the rows r = s mod stride"""
    stride = stride or S
    a = np.zeros((S, n), dtype=bool)
    for s in range(S):
        a[s, s::stride] = True
    return a
