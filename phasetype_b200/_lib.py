"""ctypes binding of libpht_b200.so (the C ABI declared in include/pht_b200.h).

The library is the product; there is no Python or CPU implementation of the hot path.
Loading fails loudly when the shared object has not been built (run
`python -m phasetype_b200.build` or `__graft_entry__.build()`).
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PHT_B200_LIB") or os.path.join(HERE, "libpht_b200.so")

# every symbol include/pht_b200.h declares (tests check the export list against the header)
SYMBOLS = [
    "LJMA_Gibbs", "pht_last_error", "pht_device_count", "pht_release_device_memory", "pht_choose_zbits", "pht_engine_create",
    "pht_engine_destroy", "pht_comm_unique_id", "pht_engine_comm_init", "pht_engine_set_theta",
    "pht_engine_get_theta", "pht_engine_run", "pht_engine_enqueue", "pht_engine_sync", "pht_engine_last_ms",
    "pht_engine_sweep_stats", "pht_engine_paths", "pht_engine_set_spectral", "pht_engine_get_model",
    "pht_engine_counters", "pht_fp64_fma_rate", "pht_engine_set_l2_flush", "pht_engine_peer_handle", "pht_engine_peer_attach", "pht_engine_round_trace", "pht_engine_set_pi", "pht_engine_get_pi", "pht_engine_pi_rows",
    "pht_engine_set_upper", "pht_engine_set_entry", "pht_engine_entry_paths",
    "pht_engine_set_chains", "pht_engine_set_chain_theta", "pht_engine_get_chain_theta", "pht_engine_chain_rows",
    "pht_engine_set_groups", "pht_engine_group_stats", "pht_engine_set_counts", "pht_engine_set_visits",
    "pht_engine_set_stage_visits", "pht_engine_set_emission", "pht_engine_get_emission", "pht_engine_emission_rows",
    "pht_engine_emission_stats",
]
PEER_HANDLE_BYTES = 128
# method 64 (include/pht_b200.h PHT_METHOD_UNIF): the uniformisation path sampler; exact, right-, interval- and
# left-censored observations, any sub-generator; delayed entry (Engine.set_entry) is this method's alone
METHOD_UNIF = 64
MAX_CHAINS = 1024            # include/pht_b200.h PHT_MAX_CHAINS: chains one METHOD_UNIF engine can run (Engine.set_chains)
MAX_GROUPS = 64              # include/pht_b200.h PHT_MAX_GROUPS: groups with their own structure (Engine.set_groups)
MAX_VISITS = 1024            # include/pht_b200.h PHT_MAX_VISITS: visits of one observation (Engine.set_visits)
MAX_STAGES = 32              # include/pht_b200.h PHT_MAX_STAGES: observed stages of stage visits (Engine.set_stage_visits)
CNT_NAMES = ["paths", "attempts", "jumps", "dens_evals", "env_updates", "brent_evals", "arms_calls",
             "metrop_rejects", "nonfinite", "deferred", "tail_rounds", "errors", "launches", "ns_lane", "ns_tail", "ns_replay",
             "ns_global", "ns_xwait", "global_rounds", "global_items"]
N_CNT = 20

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lp = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_up = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")


class Config(C.Structure):
    _fields_ = [("n", C.c_int), ("m", C.c_int), ("method", C.c_int), ("mhit", C.c_int),
                ("T", C.c_void_p), ("C", C.c_void_p), ("nu", C.c_void_p), ("zeta", C.c_void_p),
                ("seed", C.c_uint64), ("device", C.c_int), ("rank", C.c_int), ("world", C.c_int),
                ("zbits", C.c_int), ("mhrs_cap", C.c_int), ("use_graph", C.c_int)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("phasetype_b200: %s has not been built (python -m phasetype_b200.build); "
                           "there is no fallback implementation" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.pht_last_error.restype = C.c_char_p
    L.pht_device_count.restype = C.c_int
    L.pht_choose_zbits.restype = C.c_int; L.pht_choose_zbits.argtypes = [C.c_double]
    L.LJMA_Gibbs.restype = None
    L.LJMA_Gibbs.argtypes = [_ip, _ip, _ip, _ip, _ip, _dp, _dp, _ip, _dp, _dp, _ip, _ip, _dp, _ip, _dp]
    L.pht_engine_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(Config), _dp, _ip, C.c_long]
    L.pht_engine_destroy.restype = None; L.pht_engine_destroy.argtypes = [C.c_void_p]
    L.pht_comm_unique_id.argtypes = [C.c_void_p]
    L.pht_engine_comm_init.argtypes = [C.c_void_p, C.c_void_p]
    L.pht_engine_set_theta.argtypes = [C.c_void_p, _dp, C.c_uint32]
    L.pht_engine_get_theta.argtypes = [C.c_void_p, _dp]
    L.pht_engine_run.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.pht_engine_enqueue.argtypes = [C.c_void_p, C.c_int]
    L.pht_engine_sync.argtypes = [C.c_void_p]
    L.pht_engine_last_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.pht_engine_sweep_stats.argtypes = [C.c_void_p, _lp, _lp, _lp]
    L.pht_engine_paths.argtypes = [C.c_void_p, C.c_long, C.c_long, _ip, _ip, _dp]
    L.pht_engine_set_spectral.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.pht_engine_get_model.argtypes = [C.c_void_p] + [C.c_void_p] * 7
    L.pht_engine_counters.argtypes = [C.c_void_p, _up]
    L.pht_fp64_fma_rate.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.pht_engine_set_l2_flush.argtypes = [C.c_void_p, C.c_ulonglong]
    L.pht_engine_round_trace.argtypes = [C.c_void_p, _up]
    L.pht_engine_set_pi.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.pht_engine_get_pi.argtypes = [C.c_void_p, _dp]
    L.pht_engine_pi_rows.argtypes = [C.c_void_p, C.c_int, _dp]
    L.pht_engine_set_upper.argtypes = [C.c_void_p, C.c_void_p]
    L.pht_engine_set_entry.argtypes = [C.c_void_p, C.c_void_p]
    L.pht_engine_entry_paths.argtypes = [C.c_void_p, C.c_long, C.c_long, _ip, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p]
    L.pht_engine_set_chains.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.pht_engine_set_chain_theta.argtypes = [C.c_void_p, _dp, C.c_uint32]
    L.pht_engine_get_chain_theta.argtypes = [C.c_void_p, _dp]
    L.pht_engine_chain_rows.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.pht_engine_set_groups.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.pht_engine_group_stats.argtypes = [C.c_void_p, _lp, _lp, _lp]
    L.pht_engine_set_counts.argtypes = [C.c_void_p, C.c_void_p]
    L.pht_engine_set_visits.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.pht_engine_set_stage_visits.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.pht_engine_set_emission.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.pht_engine_get_emission.argtypes = [C.c_void_p, _dp]
    L.pht_engine_emission_rows.argtypes = [C.c_void_p, C.c_int, _dp]
    L.pht_engine_emission_stats.argtypes = [C.c_void_p, _lp]
    L.pht_engine_peer_handle.argtypes = [C.c_void_p, C.c_void_p]
    L.pht_engine_peer_attach.argtypes = [C.c_void_p, C.c_void_p]
    _lib = L
    return L


class EngineError(RuntimeError):
    pass


def _check(rc):
    if rc != 0:
        raise EngineError(lib().pht_last_error().decode())


class Engine:
    """One GPU's shard of a Gibbs run (thin object wrapper over the pht_engine_* calls)."""

    def __init__(self, n, T, Cmat, nu, zeta, y_local, cens_local, method, mhit=1, seed=0x5048, device=0,
                 rank=0, world=1, zbits=None, mhrs_cap=0, use_graph=True, sum_y_global=None):
        L = lib()
        self.n = int(n)
        self._T = np.ascontiguousarray(np.asarray(T, dtype=np.int32).ravel())
        self._C = np.ascontiguousarray(np.asarray(Cmat, dtype=np.float64).ravel())
        self._nu = np.ascontiguousarray(nu, dtype=np.float64)
        self._zeta = np.ascontiguousarray(zeta, dtype=np.float64)
        self.m = int(self._nu.shape[0])
        y_local = np.ascontiguousarray(y_local, dtype=np.float64)
        cens_local = np.ascontiguousarray(cens_local, dtype=np.int32)
        self.l_local = int(y_local.shape[0])
        if zbits is None and sum_y_global is None and int(world) > 1:
            # every rank must use the same fixed-point scale: a per-rank guess from the local sum can differ near a power of two
            raise EngineError("with several ranks pass sum_y_global (the sum of y over ALL ranks) or an explicit zbits")
        if zbits is None:
            zbits = L.pht_choose_zbits(float(sum_y_global if sum_y_global is not None else y_local.sum() * world))
        self.zbits = int(zbits)
        cfg = Config(self.n, self.m, int(method), int(mhit), self._T.ctypes.data, self._C.ctypes.data,
                     self._nu.ctypes.data, self._zeta.ctypes.data, int(seed), int(device), int(rank), int(world),
                     self.zbits, int(mhrs_cap), 1 if use_graph else 0)
        self._h = C.c_void_p()
        self.chains = 1
        self.groups = 1
        self.stages = 0
        _check(L.pht_engine_create(C.byref(self._h), C.byref(cfg), y_local if self.l_local else np.zeros(1),
                                   cens_local if self.l_local else np.zeros(1, dtype=np.int32), self.l_local))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().pht_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def comm_init(self, id128):
        buf = (C.c_char * 128).from_buffer_copy(bytes(id128))
        _check(lib().pht_engine_comm_init(self._h, buf))

    def peer_handle(self):
        buf = (C.c_char * PEER_HANDLE_BYTES)()
        _check(lib().pht_engine_peer_handle(self._h, buf))
        return bytes(buf.raw)

    def peer_attach(self, handles):
        """handles: the peer_handle() bytes of every rank, concatenated in rank order."""
        raw = bytes(handles)
        buf = (C.c_char * len(raw)).from_buffer_copy(raw)
        _check(lib().pht_engine_peer_attach(self._h, buf))

    def set_theta(self, theta, next_iter=1):
        _check(lib().pht_engine_set_theta(self._h, np.ascontiguousarray(theta, dtype=np.float64), int(next_iter)))

    def get_theta(self):
        out = np.zeros(self.m)
        _check(lib().pht_engine_get_theta(self._h, out))
        return out

    def run(self, nsweeps):
        out = np.zeros((int(nsweeps), self.m))
        _check(lib().pht_engine_run(self._h, int(nsweeps), out.ctypes.data if nsweeps else None))
        return out

    def enqueue(self, nsweeps):
        _check(lib().pht_engine_enqueue(self._h, int(nsweeps)))

    def sync(self):
        _check(lib().pht_engine_sync(self._h))

    def set_l2_flush(self, nbytes):
        _check(lib().pht_engine_set_l2_flush(self._h, int(nbytes)))

    def last_ms(self):
        t = C.c_float(); k = C.c_float()
        _check(lib().pht_engine_last_ms(self._h, C.byref(t), C.byref(k)))
        return t.value, k.value

    def sweep_stats(self):
        n = self.n
        N = np.zeros(n * n, dtype=np.int64); B = np.zeros(n, dtype=np.int64); z = np.zeros(n, dtype=np.int64)
        _check(lib().pht_engine_sweep_stats(self._h, N, B, z))
        return N, B, z

    def paths(self, first=0, count=None):
        n = self.n
        count = self.l_local - first if count is None else count
        B = np.zeros(count, dtype=np.int32); N = np.zeros(count * n * n, dtype=np.int32); z = np.zeros(count * n)
        _check(lib().pht_engine_paths(self._h, int(first), int(count), B, N, z))
        return B, N.reshape(count, n * n), z.reshape(count, n)

    def set_spectral(self, evals, Q, Qinv):
        if evals is None:
            _check(lib().pht_engine_set_spectral(self._h, None, None, None))
            return
        a = [np.ascontiguousarray(x, dtype=np.float64) for x in (evals, Q, Qinv)]
        _check(lib().pht_engine_set_spectral(self._h, a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data))

    def model(self):
        n = self.n
        out = {"S": np.zeros(n * n), "s": np.zeros(n), "P": np.zeros(n * n), "Pfull": np.zeros(n * (n + 1)),
               "evals": np.zeros(n), "Q": np.zeros(n * n), "Qinv": np.zeros(n * n)}
        _check(lib().pht_engine_get_model(self._h, *[out[k].ctypes.data for k in
                                                     ("S", "s", "P", "Pfull", "evals", "Q", "Qinv")]))
        return out

    def set_pi(self, pi=None, beta=None):
        a = None if pi is None else np.ascontiguousarray(pi, dtype=np.float64)
        b = None if beta is None else np.ascontiguousarray(beta, dtype=np.float64)
        _check(lib().pht_engine_set_pi(self._h, None if a is None else a.ctypes.data, None if b is None else b.ctypes.data))

    def get_pi(self):
        out = np.zeros(self.n)
        _check(lib().pht_engine_get_pi(self._h, out))
        return out

    def pi_rows(self, rows):
        out = np.zeros((int(rows), self.n))
        _check(lib().pht_engine_pi_rows(self._h, int(rows), out))
        return out

    def set_upper(self, u):
        """Interval-censored observations (methods MHRS and METHOD_UNIF): u[k] is the upper bound of local observation k's absorption time
        (+inf: none; a finite bound needs the censoring flag and u > y; METHOD_UNIF also takes y = 0, a failure before
        the first inspection); None clears the bounds.  Interval paths end by u,
        so construct the engine with sum_y_global = the sum of max(y, u) over all observations (or a zbits at most
        pht_choose_zbits of it)."""
        if u is None:
            _check(lib().pht_engine_set_upper(self._h, None))
            return
        a = np.ascontiguousarray(u, dtype=np.float64)
        if a.shape != (self.l_local,):
            raise EngineError("set_upper: %d bounds for %d local observations" % (a.size, self.l_local))
        if not self.l_local:
            a = np.full(1, np.inf)           # an empty shard still takes part (never NULL, which clears)
        _check(lib().pht_engine_set_upper(self._h, a.ctypes.data))

    def set_entry(self, a):
        """Delayed entry, or left truncation (METHOD_UNIF only): a[k] is the age at which local observation k entered the
        study (0: none; 0 <= a <= y); None clears the ages.  Each sweep then also draws, per truncated observation, the
        units of its kind lost before entry and their paths.  Those paths end by a, so construct the engine with
        sum_y_global = the sum of max(y, u) + a over all observations (or a zbits at most pht_choose_zbits of it)."""
        if a is None:
            _check(lib().pht_engine_set_entry(self._h, None))
            return
        v = np.ascontiguousarray(a, dtype=np.float64)
        if v.shape != (self.l_local,):
            raise EngineError("set_entry: %d entry ages for %d local observations" % (v.size, self.l_local))
        if not self.l_local:
            v = np.zeros(1)                  # an empty shard still takes part (never NULL, which clears)
        _check(lib().pht_engine_set_entry(self._h, v.ctypes.data))

    def entry_paths(self, first=0, count=None, paths=True):
        """Ghost counts M (count,) of local observations [first, first + count) at the current parameters, and with paths
        the ghost paths in (observation, ghost index) order: (M, B, N, z) with B (G,), N (G, n*n), z (G, n), G = M.sum()."""
        n = self.n
        count = self.l_local - first if count is None else count
        M = np.zeros(max(int(count), 1), dtype=np.int32)
        _check(lib().pht_engine_entry_paths(self._h, int(first), int(count), M, 0, None, None, None))
        M = M[:int(count)]
        if not paths:
            return M
        G = int(M.astype(np.int64).sum())
        B = np.zeros(max(G, 1), dtype=np.int32); N = np.zeros(max(G, 1) * n * n, dtype=np.int32); z = np.zeros(max(G, 1) * n)
        M2 = np.zeros(max(int(count), 1), dtype=np.int32)
        _check(lib().pht_engine_entry_paths(self._h, int(first), int(count), M2, G, B.ctypes.data, N.ctypes.data, z.ctypes.data))
        if not np.array_equal(M2[:int(count)], M):
            raise EngineError("entry_paths: ghost counts changed between two calls at the same parameters")
        return M, B[:G], N[:G * n * n].reshape(G, n * n), z[:G * n].reshape(G, n)

    def set_chains(self, chains, keys=None):
        """Several chains in this engine (METHOD_UNIF only, one rank, no entry ages): chain c draws with Philox key keys[c]
        (default: seed + c) and is bit for bit the chain of a single-chain engine with that key.  Every chain starts from
        the current theta and pi; set_theta and set_pi then set every chain, and the single-chain calls (get_theta, run,
        pi_rows, model, paths, sweep_stats) refer to chain 0.  chains = 1 returns to the single-chain engine."""
        chains = int(chains)
        k = None
        if keys is not None:
            k = np.ascontiguousarray(keys, dtype=np.uint64)
            if k.shape != (chains,):
                raise EngineError("set_chains: %d keys for %d chains" % (k.size, chains))
        _check(lib().pht_engine_set_chains(self._h, chains, None if k is None else k.ctypes.data))
        self.chains = chains

    def set_chain_theta(self, theta, next_iter=1):
        """One parameter vector per chain: theta of shape (chains, m)."""
        t = np.ascontiguousarray(theta, dtype=np.float64)
        if t.shape != (self.chains, self.m):
            raise EngineError("set_chain_theta: shape %s, expected (%d, %d)" % (t.shape, self.chains, self.m))
        _check(lib().pht_engine_set_chain_theta(self._h, t.ravel(), int(next_iter)))

    def get_chain_theta(self):
        out = np.zeros(self.chains * self.m)
        _check(lib().pht_engine_get_chain_theta(self._h, out))
        return out.reshape(self.chains, self.m)

    def run_chains(self, nsweeps):
        """nsweeps sweeps of every chain; returns the draws of theta, shape (chains, nsweeps, m)."""
        nsweeps = int(nsweeps)
        _check(lib().pht_engine_run(self._h, nsweeps, None))
        out = np.zeros((self.chains, nsweeps, self.m))
        _check(lib().pht_engine_chain_rows(self._h, nsweeps, out.ctypes.data, None))
        return out

    def chain_pi_rows(self, rows):
        """The pi draws of the last run, shape (chains, rows, n) (needs set_pi with a prior)."""
        out = np.zeros((self.chains, int(rows), self.n))
        _check(lib().pht_engine_chain_rows(self._h, int(rows), None, out.ctypes.data))
        return out

    def set_groups(self, T, Cmat=None, group=None):
        """Groups of observations with their own structure over the one parameter vector (METHOD_UNIF only, one rank, no
        entry ages with more than one group): T and Cmat shaped (G, ...), group g's T and C flattened as the constructor
        takes them; group[k] in 0..G-1 is the group of local observation k.  Every chain keeps its theta and pi; group
        g's observations are drawn on (T[g], Cmat[g]), and theta's update sums every group's cells.  T = None returns to
        the configured structure."""
        if T is None:
            _check(lib().pht_engine_set_groups(self._h, 0, None, None, None))
            self.groups = 1
            return
        t = np.asarray(T, dtype=np.int32); c = np.asarray(Cmat, dtype=np.float64)
        G, n1 = int(t.shape[0]), (self.n + 1) ** 2
        if t.size != G * n1 or c.size != G * n1:
            raise EngineError("set_groups: T %s and C %s, expected %d structures of %d entries each" % (t.shape, c.shape, G, n1))
        t = np.ascontiguousarray(t.reshape(G, n1)); c = np.ascontiguousarray(c.reshape(G, n1))
        if not G:
            t = np.zeros((1, n1), dtype=np.int32); c = np.zeros((1, n1))
        g = np.ascontiguousarray(group, dtype=np.int32)
        if g.shape != (self.l_local,):
            raise EngineError("set_groups: %d group ids for %d local observations" % (g.size, self.l_local))
        if not self.l_local:
            g = np.zeros(1, dtype=np.int32)
        _check(lib().pht_engine_set_groups(self._h, G, t.ctypes.data, c.ctypes.data, g.ctypes.data))
        self.groups = G

    def set_counts(self, counts):
        """Observations with counts (METHOD_UNIF only, one rank, no entry ages): local record k stands for counts[k] >= 0
        tied units, and the engine is bit for bit the engine on np.repeat(records, counts) (synth.tabulate builds such
        records).  Every unit's path ends by max(y, u), so construct the engine with sum_y_global = the sum of
        counts x max(y, u) over the records (or a zbits at most pht_choose_zbits of it).  None returns to plain records."""
        if counts is None:
            _check(lib().pht_engine_set_counts(self._h, None))
            return
        w = np.asarray(counts)
        if w.shape != (self.l_local,):
            raise EngineError("set_counts: %d counts for %d local records" % (w.size, self.l_local))
        if w.size and (w.min() < 0 or w.max() > 0xffffffff):
            raise EngineError("set_counts: counts must lie in 0 .. 2^32 - 1")
        w = np.ascontiguousarray(w, dtype=np.uint32)
        if not self.l_local:
            w = np.zeros(1, dtype=np.uint32)     # an empty shard still takes part (never NULL, which clears)
        _check(lib().pht_engine_set_counts(self._h, w.ctypes.data))

    def set_visits(self, offsets, t=None, mask=None):
        """Panel observations (METHOD_UNIF only, one rank, no counts): local observation k was seen at times
        t[offsets[k]:offsets[k + 1]] (increasing, within [0, y_k]) in one of the phases of mask[...] (uint32 bitmasks,
        bit c: phase c; synth.stage_masks builds stage masks).  offsets has l_local + 1 entries starting at 0.  Each path is
        then drawn given its visits too; observations without visits draw the paths they drew before.  None clears them."""
        if offsets is None:
            _check(lib().pht_engine_set_visits(self._h, None, None, None))
            self.stages = 0                  # mask visits replace stage visits
            return
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        if off.shape != (self.l_local + 1,):
            raise EngineError("set_visits: %d offsets for %d local observations (expected l_local + 1)" % (off.size, self.l_local))
        total = int(off[-1]) if off.size else 0
        tv = np.ascontiguousarray(t if t is not None else np.zeros(0), dtype=np.float64)
        mv = np.asarray(mask if mask is not None else np.zeros(0, dtype=np.uint32))
        if tv.shape != (total,) or mv.shape != (total,):
            raise EngineError("set_visits: %d times and %d masks for %d visits" % (tv.size, mv.size, total))
        if mv.size and (mv.min() < 0 or mv.max() > 0xffffffff):
            raise EngineError("set_visits: masks must lie in 0 .. 2^32 - 1")
        mv = np.ascontiguousarray(mv, dtype=np.uint32)
        tv = tv if total else np.zeros(1); mv = mv if total else np.zeros(1, dtype=np.uint32)
        _check(lib().pht_engine_set_visits(self._h, off.ctypes.data, tv.ctypes.data, mv.ctypes.data))
        self.stages = 0

    def set_stage_visits(self, E, offsets, t=None, stage=None, alpha=None):
        """Misclassified panel observations (METHOD_UNIF only, one rank, no counts): local observation k was read at times
        t[offsets[k]:offsets[k + 1]] (as set_visits) as the stages stage[...] in 0..S-1, through the emission matrix E
        (n, S): P(stage o read | phase c) = E[c, o], rows summing to 1.  alpha (n, S), when given, is a Dirichlet prior on
        E's rows (0: a structural zero, else >= 0.1, with E's support): every sweep then also draws E.  Replaces mask
        visits; offsets None clears the visits."""
        if offsets is None:
            _check(lib().pht_engine_set_stage_visits(self._h, 0, None, None, None, None, None))
            self.stages = 0
            return
        Em = np.ascontiguousarray(E, dtype=np.float64)
        if Em.ndim != 2 or Em.shape[0] != self.n:
            raise EngineError("set_stage_visits: E has shape %s, expected (%d, stages)" % (Em.shape, self.n))
        S = int(Em.shape[1])
        a = None if alpha is None else np.ascontiguousarray(alpha, dtype=np.float64)
        if a is not None and a.shape != Em.shape:
            raise EngineError("set_stage_visits: alpha has shape %s, E %s" % (a.shape, Em.shape))
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        if off.shape != (self.l_local + 1,):
            raise EngineError("set_stage_visits: %d offsets for %d local observations (expected l_local + 1)" % (off.size, self.l_local))
        total = int(off[-1]) if off.size else 0
        tv = np.ascontiguousarray(t if t is not None else np.zeros(0), dtype=np.float64)
        sv = np.asarray(stage if stage is not None else np.zeros(0, dtype=np.uint32))
        if tv.shape != (total,) or sv.shape != (total,):
            raise EngineError("set_stage_visits: %d times and %d stages for %d visits" % (tv.size, sv.size, total))
        if sv.size and (sv.min() < 0 or sv.max() > 0xffffffff):
            raise EngineError("set_stage_visits: stages must lie in 0 .. 2^32 - 1")
        sv = np.ascontiguousarray(sv, dtype=np.uint32)
        tv = tv if total else np.zeros(1); sv = sv if total else np.zeros(1, dtype=np.uint32)
        _check(lib().pht_engine_set_stage_visits(self._h, S, Em.ctypes.data, None if a is None else a.ctypes.data,
                                                 off.ctypes.data, tv.ctypes.data, sv.ctypes.data))
        self.stages = S

    def set_emission(self, E=None, alpha=None):
        """E (n, S) of every chain and / or its Dirichlet prior (None E: each chain keeps its own E; None alpha: E fixed from
        now on)."""
        S = self.stages
        Em = None if E is None else np.ascontiguousarray(E, dtype=np.float64)
        a = None if alpha is None else np.ascontiguousarray(alpha, dtype=np.float64)
        for x, what in ((Em, "E"), (a, "alpha")):
            if x is not None and S and x.shape != (self.n, S):
                raise EngineError("set_emission: %s has shape %s, expected (%d, %d)" % (what, x.shape, self.n, S))
        _check(lib().pht_engine_set_emission(self._h, None if Em is None else Em.ctypes.data, None if a is None else a.ctypes.data))

    def emission(self):
        """Chain 0's current E, shape (n, S)."""
        out = np.zeros(self.n * max(self.stages, 1))
        _check(lib().pht_engine_get_emission(self._h, out))
        return out.reshape(self.n, -1)

    def emission_rows(self, rows):
        """The E draws of the last run, shape (chains, rows, n, S) (needs alpha)."""
        S = max(self.stages, 1)
        out = np.zeros(max(self.chains * int(rows) * self.n * S, 1))
        _check(lib().pht_engine_emission_rows(self._h, int(rows), out))
        return out[:self.chains * int(rows) * self.n * S].reshape(self.chains, int(rows), self.n, S)

    def emission_stats(self):
        """K (n, S) of one sweep of chain 0 without an update: visits drawn in phase c and read as stage o."""
        K = np.zeros(self.n * max(self.stages, 1), dtype=np.int64)
        _check(lib().pht_engine_emission_stats(self._h, K))
        return K.reshape(self.n, -1)

    def group_stats(self):
        """One sweep's statistics of chain 0 per group, without an update: N (G, n*n), B (G, n), zfix (G, n); their sum
        over the groups is sweep_stats()."""
        n, G = self.n, self.groups
        N = np.zeros(G * n * n, dtype=np.int64); B = np.zeros(G * n, dtype=np.int64); z = np.zeros(G * n, dtype=np.int64)
        _check(lib().pht_engine_group_stats(self._h, N, B, z))
        return N.reshape(G, n * n), B.reshape(G, n), z.reshape(G, n)

    def round_trace(self):
        """(48, 8) array: per tail round number, ns search / ns barrier / ns advance / sum of pending / sum of K / attempts run /
        attempts the sequential sampler needs of this round / jump-steps run."""
        t = np.zeros(48 * 8, dtype=np.uint64)
        _check(lib().pht_engine_round_trace(self._h, t))
        return t.reshape(48, 8)

    def counters(self):
        c = np.zeros(N_CNT, dtype=np.uint64)
        _check(lib().pht_engine_counters(self._h, c))
        return {k: int(c[i]) for i, k in enumerate(CNT_NAMES)}


def fp64_fma_rate(device=0):
    r = C.c_double()
    if lib().pht_fp64_fma_rate(int(device), C.byref(r)) != 0:
        raise EngineError("FP64 microbenchmark failed (no CUDA device?)")
    return r.value
