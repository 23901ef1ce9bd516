"""ctypes bindings for the checkers in oracle/ (TEST INFRASTRUCTURE ONLY).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module; nothing under phasetype_b200/ does.

Two libraries:
  * oracle/_build/libphtoracle.so -- the CPU restatement (pht_oracle.c), built by `make oracle`;
  * oracle/_ref/libphtref.so      -- the unmodified reference C + R stand-in, built by `make ref`
                                     where PHT_REFERENCE_SRC names an upstream PhaseType source tree
                                     (https://github.com/louisaslett/PhaseType); without it the tests that
                                     compare against the reference skip.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "_build", "libphtoracle.so")
REF_SO = os.path.join(HERE, "_ref", "libphtref.so")
REF_LIBM_SO = os.path.join(HERE, "_ref", "libphtref_libm.so")
REG_SO = os.path.join(HERE, "_ref", "PhaseType_reg.so")
REFERENCE_ROOT = os.environ.get("PHT_REFERENCE_SRC", "")

N_COUNTERS = 16
COUNTER_NAMES = ["paths", "attempts", "jumps", "dens_evals", "env_updates", "brent_evals",
                 "arms_calls", "metrop_rejects", "nonfinite"]

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lp = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_up = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")


def build(target="all"):
    """Compile the checkers (gcc).  `ref` is skipped when no reference tree is given (PHT_REFERENCE_SRC)."""
    targets = ["oracle"]
    if target in ("all", "ref") and REFERENCE_ROOT and os.path.isdir(os.path.join(REFERENCE_ROOT, "src")):
        targets.append("ref")
        targets.append("ref-libm")
        if os.path.exists(os.path.join(HERE, "..", "phasetype_b200", "libpht_b200.so")):
            targets.append("reg")
    ref = ["REF=" + os.path.abspath(REFERENCE_ROOT)] if REFERENCE_ROOT else []
    subprocess.run(["make", "-s", "-C", HERE] + ref + targets, check=True)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def embedded(S, s):
    """P, Pfull exactly as src/PHT_MCMC_Aslett.c:280-297 (column-major n*n and n*(n+1))."""
    lib = oracle()
    S = _f64(S); s = _f64(s); n = s.shape[0]
    P = np.zeros(n * n); Pfull = np.zeros(n * (n + 1))
    lib.pho_embedded(n, S, s, P, Pfull)
    return P, Pfull


class _Lib:
    def __init__(self, path):
        if not os.path.exists(path):
            raise FileNotFoundError(path + " is missing: run `make -C oracle`")
        self.path = path
        self.lib = C.CDLL(path)

    def __getattr__(self, name):
        return getattr(self.lib, name)


_oracle = None
_ref = None
_ref_libm = None


def oracle():
    global _oracle
    if _oracle is None:
        o = _Lib(ORACLE_SO)
        L = o.lib
        L.pho_exp.restype = C.c_double; L.pho_exp.argtypes = [C.c_double]
        L.pho_log.restype = C.c_double; L.pho_log.argtypes = [C.c_double]
        L.pho_exp_general.restype = C.c_double; L.pho_exp_general.argtypes = [C.c_double]
        L.pho_unif_at.restype = C.c_double
        L.pho_unif_at.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.pho_rgamma_at.restype = C.c_double
        L.pho_rgamma_at.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_double, C.c_double]
        L.pho_embedded.argtypes = [C.c_int, _dp, _dp, _dp, _dp]
        L.pho_set_pi.argtypes = [C.c_void_p, C.c_int]; L.pho_set_pi.restype = None
        L.pho_mhrs_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                     _dp, _dp, _dp, C.c_int, _ip, _ip, _dp, _up]
        for f in ("pho_dcs_paths", "pho_ecs_paths", "pho_eigen", "pho_gibbs", "pho_sweep_stats", "pho_update",
                  "pho_choose_zbits"):
            if not hasattr(L, f):
                continue
        if hasattr(L, "pho_eigen"):
            L.pho_eigen.argtypes = [C.c_int, _dp, _dp, _dp, _dp, _dp]
        if hasattr(L, "pho_eigen_native"):
            L.pho_eigen_native.argtypes = [C.c_int, _dp, _dp, _dp, _dp]
        if hasattr(L, "pho_dcs_paths"):
            L.pho_dcs_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, C.c_int,
                                        _dp, _dp, _dp, _dp, _dp, _ip, _ip, _dp, _up]
        if hasattr(L, "pho_ecs_paths"):
            L.pho_ecs_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                        _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _ip, _dp, _up]
        L.pho_mhs_hobolth_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                            _dp, _dp, _dp, _dp, _dp, C.c_int, _ip, _ip, _dp, _up]
        L.pho_mhs_aslett_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                           _dp, _dp, _dp, _dp, _dp, _dp, _dp, C.c_int, _ip, _ip, _dp, _up]
        if hasattr(L, "pho_choose_zbits"):
            L.pho_choose_zbits.restype = C.c_int; L.pho_choose_zbits.argtypes = [C.c_double]
        if hasattr(L, "pho_gibbs"):
            L.pho_gibbs.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp, _ip, _dp,
                                    _dp, C.c_long, _ip, _dp, _dp, _up]
        if hasattr(L, "pho_sweep_stats"):
            L.pho_sweep_stats.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _ip, _dp,
                                          _dp, _dp, C.c_long, _ip, C.c_int, C.c_int, C.c_int, _lp, _lp, _lp, _up]
        if hasattr(L, "pho_update"):
            L.pho_update.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, _dp, _dp, _ip, _dp, C.c_int,
                                     _lp, _lp, _dp]
        _oracle = o
    return _oracle


def have_ref():
    return os.path.exists(REF_SO)


def have_ref_libm():
    return os.path.exists(REF_LIBM_SO)


def ref(libm=False):
    """libm=True: the reference built with the platform's exp/log and OpenBLAS (`make ref-libm`)."""
    global _ref, _ref_libm
    if libm:
        if _ref_libm is None:
            _ref_libm = _load_ref(REF_LIBM_SO)
        return _ref_libm
    if _ref is None:
        _ref = _load_ref(REF_SO)
    return _ref


def _load_ref(path):
    if True:
        r = _Lib(path)
        L = r.lib
        L.phtref_mhrs_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                        _dp, _dp, _dp, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, _up]
        L.phtref_ecs_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                       _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp,
                                       C.c_void_p, C.c_void_p, C.c_void_p, _up]
        L.phtref_dcs_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                       _dp, _dp, _dp, _dp, _dp, C.c_void_p, C.c_void_p, C.c_void_p, _up]
        L.phtref_eigen.argtypes = [C.c_int, _dp, _dp, _dp, _dp]
        if hasattr(L, "phtref_mhs_hobolth_paths"):
            L.phtref_mhs_hobolth_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                                   _dp, _dp, _dp, _dp, _dp, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, _up]
            L.phtref_mhs_aslett_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_int,
                                                  _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, C.c_int,
                                                  C.c_void_p, C.c_void_p, C.c_void_p, _up]
        if hasattr(L, "phtref_set_pi"):
            L.phtref_set_pi.argtypes = [C.c_void_p, C.c_int]; L.phtref_set_pi.restype = None
        L.phtref_gibbs.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp,
                                   _ip, _dp, _dp, C.c_int, _ip, _dp, _dp]
    return r


def _out(count, n, want):
    if not want:
        return None, None, None
    return (np.zeros(count, dtype=np.int32), np.zeros(count * n * n, dtype=np.int32),
            np.zeros(count * n, dtype=np.float64))


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _counters(c):
    return {k: int(c[i]) for i, k in enumerate(COUNTER_NAMES)}


def mhrs_paths(impl, seed, it, y, cens, S, s, mhit=1, obs0=0, stride=1, want=True):
    """Per-observation (B[count], N[count,n*n], z[count,n]) + counters from `impl` in {"oracle","ref"}."""
    y = _f64(y); cens = _i32(cens); S = _f64(S); s = _f64(s)
    n = s.shape[0]; count = y.shape[0]
    P, Pfull = embedded(S, s)
    cnt = np.zeros(N_COUNTERS, dtype=np.uint64)
    B, N, z = _out(count, n, want)
    if impl == "oracle":
        if B is None:
            B, N, z = _out(count, n, True)
        rc = oracle().pho_mhrs_paths(seed, it, obs0, stride, count, y, cens, n, S, s, Pfull, mhit, B, N, z, cnt)
        counters = _counters(cnt)
    else:
        rc = ref(impl == "ref_libm").phtref_mhrs_paths(seed, it, obs0, stride, count, y, cens, n, S.copy(), s.copy(), Pfull, mhit,
                                     _ptr(B), _ptr(N), _ptr(z), cnt)
        counters = {"paths": count, "attempts": int(cnt[1]), "jumps": int(cnt[4]), "uniforms": int(cnt[0])}
    if rc != 0:
        raise RuntimeError("%s mhrs_paths failed rc=%d" % (impl, rc))
    if B is None:
        return None, None, None, counters
    return B, N.reshape(count, n * n), z.reshape(count, n), counters


def eigen(impl, S, n):
    """(evals, Q, Qinv) of the column-major n x n matrix S, through LAPACK as the reference does (src/utility.c:87-129)."""
    S = _f64(S)
    ev = np.zeros(n); Q = np.zeros(n * n); Qi = np.zeros(n * n)
    if impl == "native":
        rc = oracle().pho_eigen_native(n, S, ev, Q, Qi)
        if rc != 0:
            raise ValueError("pht_eigen_real status %d (1 = no convergence, 2 = complex pair, 4 = singular Q)" % rc)
    elif impl == "oracle":
        im = np.zeros(n)
        rc = oracle().pho_eigen(n, S, ev, im, Q, Qi)
        if rc != 0:
            raise RuntimeError("pho_eigen failed rc=%d" % rc)
        if (im != 0).any():
            raise ValueError("complex spectrum: the reference's spectral samplers are not valid for this S")
    else:
        rc = ref().phtref_eigen(n, S.copy(), ev, Q, Qi)
        if rc != 0:
            raise RuntimeError("phtref_eigen failed rc=%d" % rc)
    return ev, Q, Qi


def spectral_paths(impl, method, seed, it, y, cens, S, s, obs0=0, stride=1, want=True, spectral=None):
    """ECS / DCS per-observation statistics from `impl` in {"oracle","ref"}.  `spectral` = (evals, Q, Qinv)
    overrides the LAPACK decomposition (both implementations then consume identical numbers)."""
    y = _f64(y); cens = _i32(cens); S = _f64(S); s = _f64(s)
    n = s.shape[0]; count = y.shape[0]
    ev, Q, Qi = spectral if spectral is not None else eigen("oracle", S, n)
    ev = _f64(ev); Q = _f64(Q); Qi = _f64(Qi)
    P, Pfull = embedded(S, s)
    cnt = np.zeros(N_COUNTERS, dtype=np.uint64)
    B, N, z = _out(count, n, True if impl == "oracle" else want)
    if method == "DCS":
        if impl == "oracle":
            rc = oracle().pho_dcs_paths(seed, it, obs0, stride, count, y, n, S, s, ev, Q, Qi, B, N, z, cnt)
        else:
            rc = ref(impl == "ref_libm").phtref_dcs_paths(seed, it, obs0, stride, count, y, cens, n, S.copy(), s.copy(), ev.copy(), Q.copy(),
                                        Qi.copy(), _ptr(B), _ptr(N), _ptr(z), cnt)
    elif method == "ECS":
        Qm = Qi.reshape(n, n, order="F")
        # Q^-1 s and Q^-1 1 in the reference BLAS order (src/PHT_MCMC_Aslett.c:331-332: dgemv 'N')
        Qinv_s = np.zeros(n); Qinv_1 = np.zeros(n)
        for j in range(n):
            Qinv_s += s[j] * Qm[:, j]
            Qinv_1 += 1.0 * Qm[:, j]
        if impl == "oracle":
            rc = oracle().pho_ecs_paths(seed, it, obs0, stride, count, y, cens, n, S, s, P, Pfull, ev, Q, Qinv_s, Qinv_1,
                                        B, N, z, cnt)
        else:
            rc = ref(impl == "ref_libm").phtref_ecs_paths(seed, it, obs0, stride, count, y, cens, n, S.copy(), s.copy(), P.copy(), Pfull.copy(),
                                        ev.copy(), Q.copy(), Qinv_s, Qinv_1, _ptr(B), _ptr(N), _ptr(z), cnt)
    else:
        raise ValueError(method)
    if rc != 0:
        raise RuntimeError("%s %s paths failed rc=%d" % (impl, method, rc))
    counters = _counters(cnt) if impl == "oracle" else {"paths": count, "uniforms": int(cnt[0]), "jumps": int(cnt[4])}
    if B is None:
        return None, None, None, counters
    return B, N.reshape(count, n * n), z.reshape(count, n), counters


def mh_variant_paths(impl, method, seed, it, y, cens, S, s, mhit=1, obs0=0, stride=1, spectral=None):
    """The two MH variants the reference compiles but never dispatches (SURVEY 8(f)1): method "MHS_HOBOLTH"
    (LJMA_MHsample_Hobolth) or "MHS_ASLETT" (LJMA_MHsample_Aslett, reverse = 0), per-observation statistics from
    `impl` in {"oracle", "ref"}."""
    y = _f64(y); cens = _i32(cens); S = _f64(S); s = _f64(s)
    n = s.shape[0]; count = y.shape[0]
    ev, Q, Qi = spectral if spectral is not None else eigen("oracle", S, n)
    ev = _f64(ev); Q = _f64(Q); Qi = _f64(Qi)
    P, Pfull = embedded(S, s)
    cnt = np.zeros(N_COUNTERS, dtype=np.uint64)
    B, N, z = _out(count, n, True)
    if method == "MHS_HOBOLTH":
        if impl == "oracle":
            rc = oracle().pho_mhs_hobolth_paths(seed, it, obs0, stride, count, y, cens, n, S, s, ev, Q, Qi, mhit, B, N, z, cnt)
        else:
            rc = ref().phtref_mhs_hobolth_paths(seed, it, obs0, stride, count, y, cens, n, S.copy(), s.copy(), ev.copy(), Q.copy(),
                                                Qi.copy(), mhit, _ptr(B), _ptr(N), _ptr(z), cnt)
    elif method == "MHS_ASLETT":
        Qm = Qi.reshape(n, n, order="F")
        Qinv_1 = np.zeros(n)
        for j in range(n):
            Qinv_1 += 1.0 * Qm[:, j]
        if impl == "oracle":
            rc = oracle().pho_mhs_aslett_paths(seed, it, obs0, stride, count, y, cens, n, S, s, P, Pfull, ev, Q, Qinv_1, mhit, B, N, z, cnt)
        else:
            rc = ref().phtref_mhs_aslett_paths(seed, it, obs0, stride, count, y, cens, n, S.copy(), s.copy(), P.copy(), Pfull.copy(),
                                               ev.copy(), Q.copy(), Qinv_1, Qi.copy(), mhit, _ptr(B), _ptr(N), _ptr(z), cnt)
    else:
        raise ValueError(method)
    if rc != 0:
        raise RuntimeError("%s %s paths failed rc=%d" % (impl, method, rc))
    counters = _counters(cnt) if impl == "oracle" else {"paths": count, "uniforms": int(cnt[0]), "jumps": int(cnt[4])}
    return B, N.reshape(count, n * n), z.reshape(count, n), counters


def set_pi(pi=None):
    """Start distribution for the *_paths functions of both checkers (None: the reference's e1)."""
    a = None if pi is None else _f64(pi)
    n = 0 if a is None else a.shape[0]
    oracle().lib.pho_set_pi(_ptr(a), n)
    if have_ref():
        ref().lib.phtref_set_pi(_ptr(a), n)
    if have_ref_libm() and hasattr(ref(True).lib, "phtref_set_pi"):
        ref(True).lib.phtref_set_pi(_ptr(a), n)


def rgamma_at(seed, it, sub, shape, scale):
    return float(oracle().pho_rgamma_at(int(seed), int(it), int(sub), float(shape), float(scale)))


def choose_zbits(sum_y):
    return int(oracle().pho_choose_zbits(float(sum_y)))


def sweep_stats(seed, it, first, mhit, method, n, T, Cm, theta, y, cens, rank=0, world=1, zbits=None):
    """Packed sufficient statistics (N int64 n*n, B int64 n, z int64 fixed point) of one sweep for the shard
    {i : i % world == rank}, computed by the CPU restatement with the engine's own spectral solver."""
    y = _f64(y); cens = _i32(cens); theta = _f64(theta); T = _i32(np.asarray(T).ravel()); Cm = _f64(np.asarray(Cm).ravel())
    if zbits is None:
        zbits = choose_zbits(y.sum())
    N = np.zeros(n * n, dtype=np.int64); B = np.zeros(n, dtype=np.int64); z = np.zeros(n, dtype=np.int64)
    cnt = np.zeros(N_COUNTERS, dtype=np.uint64)
    rc = oracle().pho_sweep_stats(seed, it, 1 if first else 0, mhit, method, n, theta.shape[0], T, Cm, theta, y, y.shape[0], cens,
                                  rank, world, zbits, N, B, z, cnt)
    if rc != 0:
        raise RuntimeError("pho_sweep_stats failed rc=%d" % rc)
    return N, B, z, _counters(cnt)


def update(seed, it, n, nu, zeta, T, Cm, zbits, N, zfix):
    nu = _f64(nu); zeta = _f64(zeta); T = _i32(np.asarray(T).ravel()); Cm = _f64(np.asarray(Cm).ravel())
    out = np.zeros(nu.shape[0])
    oracle().pho_update(seed, it, n, nu.shape[0], nu, zeta, T, Cm, zbits, np.ascontiguousarray(N, dtype=np.int64),
                        np.ascontiguousarray(zfix, dtype=np.int64), out)
    return out


def gibbs(seed, it, mhit, method, n, nu, zeta, T, Cm, y, cens, start):
    """The whole chain from the CPU restatement: (it, m) array like LJMA_Gibbs's res."""
    nu = _f64(nu); zeta = _f64(zeta); T = _i32(np.asarray(T).ravel()); Cm = _f64(np.asarray(Cm).ravel())
    y = _f64(y); cens = _i32(cens); m = nu.shape[0]
    start = _f64(np.atleast_1d(start))
    if start.shape[0] < m:
        start = np.concatenate([start, np.zeros(m - start.shape[0])])
    res = np.zeros(it * m); cnt = np.zeros(N_COUNTERS, dtype=np.uint64)
    rc = oracle().pho_gibbs(seed, it, mhit, method, n, m, nu, zeta, T, Cm, y, y.shape[0], cens, start, res, cnt)
    if rc != 0:
        raise RuntimeError("pho_gibbs failed rc=%d" % rc)
    return res.reshape(m, it).T.copy(), _counters(cnt)


def ref_gibbs(seed, keyed, it, mhit, method, n, nu, zeta, T, Cm, y, cens, start):
    """The reference's own LJMA_Gibbs (unmodified C + R stand-in).  keyed=True (ECS/DCS) maps path p of sweep i
    to Philox stream (i, p); otherwise one sequential stream."""
    nu = _f64(nu).copy(); zeta = _f64(zeta).copy(); T = _i32(np.asarray(T).ravel()).copy(); Cm = _f64(np.asarray(Cm).ravel()).copy()
    y = _f64(y).copy(); cens = _i32(cens).copy(); m = nu.shape[0]
    start = _f64(np.atleast_1d(start))
    if start.shape[0] < m:
        start = np.concatenate([start, np.zeros(m - start.shape[0])])
    res = np.zeros(it * m)
    ref().phtref_gibbs(seed, 1 if keyed else 0, it, mhit, method, n, m, nu, zeta, T, Cm, y, y.shape[0], cens, start.copy(), res)
    return res.reshape(m, it).T.copy()
