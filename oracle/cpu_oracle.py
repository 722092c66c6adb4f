"""ctypes front-end of oracle/cpu/libark_cpu.so -- TEST INFRASTRUCTURE ONLY
(see the header of oracle/cpu/ark_cpu.cpp).  Array conventions are those of
include/b200zk.h: uint64 limb arrays, Fr/Fq in Montgomery form, MSM scalars
canonical."""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "cpu", "libark_cpu.so")
_lib = None
vp = ctypes.c_void_p


_STAMP = os.path.join(_HERE, "cpu", "libark_cpu.host")


def _host_signature():
    """-march=native ties the binary to the CPU it was built on (BASELINE.md: the CPU baseline is
    compiled for the host it is timed on): the ISA flag set of this machine."""
    import hashlib
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return hashlib.sha256(" ".join(sorted(line.split(":", 1)[1].split())).encode()).hexdigest()[:16]
    except OSError:
        pass
    return "unknown"


def build(force=False):
    """make -C oracle; rebuilt when the library was compiled on a different CPU (the .so travels to the
    GPU box with the repo snapshot, the box has the same toolchain)."""
    sig = _host_signature()
    have = open(_STAMP).read().strip() if os.path.exists(_STAMP) else ""
    if force or have != sig:
        subprocess.run(["make", "-C", _HERE, "-s", "clean"], check=True)
    subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    with open(_STAMP, "w") as f:
        f.write(sig)
    return _LIB_PATH


def _in_tree_current():
    """True when build() made the in-tree library on a CPU with this one's ISA flags, after the last source edit."""
    try:
        with open(_STAMP) as f:
            if f.read().strip() != _host_signature():
                return False
        return os.path.getmtime(_LIB_PATH) >= os.path.getmtime(os.path.join(_HERE, "cpu", "ark_cpu.cpp"))
    except OSError:
        return False


def _load():
    """The in-tree library when it is current; otherwise a private build in a temporary directory, so that
    loading never writes into the tree (bench.py may run from a read-only checkout)."""
    if _in_tree_current():
        return ctypes.CDLL(_LIB_PATH)
    tmp = tempfile.mkdtemp(prefix="ark_cpu_")
    try:
        path = os.path.join(tmp, "libark_cpu.so")
        subprocess.run(["make", "-C", _HERE, "-s", "ARK_CPU_LIB=" + path], check=True)
        return ctypes.CDLL(path)               # stays mapped after the directory is removed
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def lib():
    global _lib
    if _lib is None:
        L = _load()
        L.ark_cpu_set_threads.argtypes = [ctypes.c_int]
        L.ark_cpu_hardware_threads.restype = ctypes.c_int
        L.ark_cpu_ntt.argtypes = [vp, ctypes.c_uint32, ctypes.c_int, vp]
        L.ark_cpu_witness_map.argtypes = [vp, vp, vp, ctypes.c_uint32, vp]
        L.ark_cpu_msm_g1.argtypes = [vp, vp, vp, ctypes.c_uint64, vp]
        L.ark_cpu_msm_g1.restype = ctypes.c_int
        L.ark_cpu_msm_g2.argtypes = [vp, vp, vp, ctypes.c_uint64, vp]
        L.ark_cpu_msm_g2.restype = ctypes.c_int
        L.ark_cpu_pk_new.restype = vp
        L.ark_cpu_pk_new.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32] + [vp] * 15
        L.ark_cpu_pk_free.argtypes = [vp]
        L.ark_cpu_prove.argtypes = [vp] * 8
        L.ark_cpu_groth16_setup.restype = ctypes.c_int
        L.ark_cpu_groth16_setup.argtypes = [ctypes.c_uint64] * 3 + [vp] * 30
        L.ark_cpu_constraint_evals.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32] + [vp] * 13
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(vp) if a is not None else None


def _c(a, dt=np.uint64):
    return np.ascontiguousarray(a, dtype=dt) if a is not None else None


def hardware_threads():
    return lib().ark_cpu_hardware_threads()


def set_threads(t):
    lib().ark_cpu_set_threads(int(t))


def ntt(data, inverse=False, coset_gen=None):
    a = _c(data).copy()
    n = a.shape[0]
    g = _c(coset_gen)
    lib().ark_cpu_ntt(_p(a), n.bit_length() - 1, int(inverse), _p(g))
    return a


def witness_map(a, b, c):
    a, b, c = _c(a).copy(), _c(b).copy(), _c(c).copy()
    n = a.shape[0]
    h = np.empty_like(a)
    lib().ark_cpu_witness_map(_p(a), _p(b), _p(c), n.bit_length() - 1, _p(h))
    return h


def msm_g1(bases, scalars, inf=None):
    bases, scalars, inf = _c(bases), _c(scalars), _c(inf, np.uint8)
    n = min(bases.shape[0], scalars.shape[0])
    out = np.zeros(12, dtype=np.uint64)
    is_inf = lib().ark_cpu_msm_g1(_p(bases), _p(inf), _p(scalars), n, _p(out))
    return out, bool(is_inf)


def msm_g2(bases, scalars, inf=None):
    bases, scalars, inf = _c(bases), _c(scalars), _c(inf, np.uint8)
    n = min(bases.shape[0], scalars.shape[0])
    out = np.zeros(24, dtype=np.uint64)
    is_inf = lib().ark_cpu_msm_g2(_p(bases), _p(inf), _p(scalars), n, _p(out))
    return out, bool(is_inf)


class CpuProvingKey:
    """Holds an ark_cpu_pk built from the same limb arrays a b2z_pk_desc takes."""

    def __init__(self, num_variables, num_instance, domain_size, a, b1, b2, h, l, alpha, beta1, delta1, beta2, delta2):
        self._keep = []

        def q(pair):
            arr, inf = _c(pair[0]), _c(pair[1], np.uint8)
            self._keep += [arr, inf]
            return _p(arr), _p(inf)

        def one(x):
            x = _c(x)
            self._keep.append(x)
            return _p(x)

        args = [num_variables, num_instance, domain_size.bit_length() - 1]
        for pair in (a, b1, b2, h, l):
            args += list(q(pair))
        args += [one(alpha), one(beta1), one(delta1), one(beta2), one(delta2)]
        self.domain_size = domain_size
        self.handle = lib().ark_cpu_pk_new(*args)

    def prove(self, a, b, c, z, r_mont, s_mont):
        a, b, c, z = _c(a).copy(), _c(b).copy(), _c(c).copy(), _c(z)
        r_mont, s_mont = _c(r_mont), _c(s_mont)
        out = np.zeros(192, dtype=np.uint8)
        lib().ark_cpu_prove(self.handle, _p(a), _p(b), _p(c), _p(z), _p(r_mont), _p(s_mont), _p(out))
        return out.tobytes()

    def __del__(self):
        try:
            if self.handle:
                lib().ark_cpu_pk_free(self.handle)
                self.handle = None
        except Exception:
            pass


def _gen_limbs():
    from oracle import bls12_381 as O
    g1 = np.array(O.int_to_limbs(O.fq_to_mont(O.G1_GEN[0]), 6) + O.int_to_limbs(O.fq_to_mont(O.G1_GEN[1]), 6),
                  dtype=np.uint64)
    (x0, x1), (y0, y1) = O.G2_GEN
    g2 = np.array(sum((O.int_to_limbs(O.fq_to_mont(v), 6) for v in (x0, x1, y0, y1)), []), dtype=np.uint64)
    return g1, g2


class CpuKey:
    """Arrays of a Groth16 key in the b2z_pk_desc layout (limbs ndarray, identity bitmap) + the vk extras."""


def groth16_setup(csr_a, csr_b, csr_c, num_constraints, num_instance, num_variables, toxic):
    """ark-groth16 generate_parameters_with_qap on the CPU (standard generators, caller-supplied toxic waste
    alpha, beta, gamma, delta, tau as ints).  csr_*: (row_ptr uint64, cols uint32, coeffs (nnz, 4) Montgomery)."""
    nc, l, m = int(num_constraints), int(num_instance), int(num_variables)
    n = 1
    while n < nc + l:
        n <<= 1
    mats = []
    for rp, ci, cf in (csr_a, csr_b, csr_c):
        mats += [_c(rp), _c(ci, np.uint32), _c(cf)]
    tox = np.frombuffer(b"".join(int(t).to_bytes(32, "little") for t in toxic), dtype=np.uint64).copy()
    g1, g2 = _gen_limbs()
    k = CpuKey()
    k.num_variables, k.num_instance, k.domain_size = m, l, n
    z1 = lambda cnt: (np.zeros((cnt, 12), np.uint64), np.zeros((cnt + 7) // 8 + 1, np.uint8))
    z2 = lambda cnt: (np.zeros((cnt, 24), np.uint64), np.zeros((cnt + 7) // 8 + 1, np.uint8))
    k.a_query, k.b_g1_query, k.b_g2_query, k.h_query, k.l_query = z1(m), z1(m), z2(m), z1(n - 1), z1(m - l)
    k.gamma_abc_g1 = z1(l)
    k.alpha_g1, k.beta_g1, k.delta_g1 = (np.zeros(12, np.uint64) for _ in range(3))
    k.beta_g2, k.gamma_g2, k.delta_g2 = (np.zeros(24, np.uint64) for _ in range(3))
    args = [nc, l, m] + [_p(x) for x in mats] + [_p(tox), _p(g1), _p(g2)]
    for pair in (k.a_query, k.b_g1_query, k.b_g2_query, k.h_query, k.l_query):
        args += [_p(pair[0]), _p(pair[1])]
    args += [_p(x) for x in (k.alpha_g1, k.beta_g1, k.delta_g1, k.beta_g2, k.gamma_g2, k.delta_g2)]
    args += [_p(k.gamma_abc_g1[0]), _p(k.gamma_abc_g1[1])]
    st = lib().ark_cpu_groth16_setup(*args)
    if st != 0:
        raise ValueError("ark_cpu_groth16_setup failed (%d)" % st)
    return k


def constraint_evals(csr_a, csr_b, csr_c, num_constraints, num_instance, z_mont):
    """a, b, c evaluation vectors of witness_map_from_matrices (Montgomery limbs, domain size)."""
    nc, l = int(num_constraints), int(num_instance)
    log_n = max(0, (nc + l - 1).bit_length())
    n = 1 << log_n
    mats = []
    for rp, ci, cf in (csr_a, csr_b, csr_c):
        mats += [_c(rp), _c(ci, np.uint32), _c(cf)]
    z = _c(z_mont)
    a, b, c = (np.zeros((n, 4), np.uint64) for _ in range(3))
    lib().ark_cpu_constraint_evals(nc, l, log_n, *[_p(x) for x in mats], _p(z), _p(a), _p(b), _p(c))
    return a, b, c


def proving_key_of(k):
    return CpuProvingKey(k.num_variables, k.num_instance, k.domain_size, k.a_query, k.b_g1_query, k.b_g2_query,
                         k.h_query, k.l_query, k.alpha_g1, k.beta_g1, k.delta_g1, k.beta_g2, k.delta_g2)
