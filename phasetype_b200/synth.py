"""Synthetic workloads of the five BASELINE.json configs (SURVEY.md section 8(d)), as
LJMA_Gibbs argument vectors.  Host-side numpy only; everything is seeded so every rank of a
multi-GPU run regenerates the same global data set and takes its strided shard.

C1  3-phase package example (man/PhaseType-package.Rd:39), l = 100, it = 1000
C2  4-phase Coxian, forward rates 1.0 + 0.37 i, early exit 0.3, last exit 1.5, l = 1e6, exact
C3  8-phase dense, rates iid U(0.2, 1.2) (symmetrised for ECS/DCS so the spectrum is real), l = 1e7, 20 % censored
C4  16 up-states of a repairable series-parallel system with tied F / R rates, l = 1e7
C5  32-phase dense, l = 1e8
Priors nu = 2, zeta = 2 / theta_true; start = theta_true.
"""
import numpy as np

SEED0 = 0x5048


class Workload:
    def __init__(self, name, n, T, C, theta, nu, zeta, y, censored, R, s):
        self.name = name; self.n = n; self.T = T; self.C = C; self.theta = theta
        self.nu = nu; self.zeta = zeta; self.y = y; self.censored = censored; self.R = R; self.s = s
        self.m = int(theta.shape[0])

    @property
    def l(self):
        return int(self.y.shape[0])

    def shard(self, rank, world):
        return self.y[rank::world], self.censored[rank::world]


def simulate_pht(R, s, size, rng, chunk=1 << 20):
    """Absorption times of the CTMC with off-diagonal rates R and exit rates s, started in state 0
    (vectorised over paths: one numpy pass per jump over the still-active paths)."""
    n = s.shape[0]
    rate = R.sum(1) + s
    cum = np.cumsum(np.concatenate([R, s[:, None]], axis=1) / rate[:, None], axis=1)
    cum[:, -1] = 1.0
    out = np.empty(size)
    for lo in range(0, size, chunk):
        k = min(chunk, size - lo)
        t = np.zeros(k); state = np.zeros(k, dtype=np.int64); alive = np.arange(k)
        while alive.size:
            st = state[alive]
            t[alive] += rng.exponential(1.0, alive.size) / rate[st]
            u = rng.random(alive.size)
            nxt = (u[:, None] >= cum[st]).sum(1)
            state[alive] = nxt
            alive = alive[nxt < n]
        out[lo:lo + k] = t
    return out


def inspection(R, s, l, spacing, k, rng):
    """Inspection data (interval censoring): absorption times T of the CTMC (R, s) started in state 0, seen only at the
    inspections spacing, 2 spacing, ..., k spacing.  A unit found failed at inspection i (T in ((i-1) spacing, i spacing])
    gives the interval y = (i-1) spacing, u = i spacing (y = 1e-12 before the first inspection: the sampler needs y > 0);
    a unit still working at the last inspection is right-censored there (u = +inf).  Returns (y, u, censored, T)."""
    t = simulate_pht(R, s, l, rng)
    i = np.ceil(t / spacing)
    failed = i <= k
    y = np.where(failed, np.maximum((i - 1) * spacing, 1e-12), k * spacing)
    u = np.where(failed, i * spacing, np.inf)
    return y, u, np.ones(l, dtype=np.int32), t


def stage_masks(stage_of_phase):
    """The uint32 phase mask of every stage: stage_of_phase[c] is the observed stage of phase c (stages 0, 1, ...); entry k
    of the result has bit c set for every phase c of stage k."""
    st = np.asarray(stage_of_phase, dtype=np.int64)
    return np.array([sum(1 << int(c) for c in np.flatnonzero(st == k)) for k in range(int(st.max()) + 1)], dtype=np.uint32)


def panel(R, s, l, spacing, k, stage_of_phase, rng, censor=None):
    """Panel data (Engine.set_visits): l units of the CTMC (R, s) started in state 0, inspected at spacing, 2 spacing, ...,
    up to k times while still working; each inspection records the mask of the stage (stage_masks) of the phase occupied
    then.  The absorption time is exact; censor(l, rng), when given, draws censoring times: a unit still working then is
    right-censored there, and only inspections up to it are kept.  Returns (y, censored, offsets, t, mask)."""
    n = s.shape[0]
    masks = stage_masks(stage_of_phase)
    stage = np.asarray(stage_of_phase, dtype=np.int64)
    rate = R.sum(1) + s
    cum = np.cumsum(np.concatenate([R, s[:, None]], axis=1) / rate[:, None], axis=1)
    cum[:, -1] = 1.0
    end = np.full(l, np.inf) if censor is None else np.asarray(censor(l, rng), dtype=np.float64)
    ins = spacing * np.arange(1, k + 1)
    seen = np.full((l, k), -1, dtype=np.int64)           # phase at each inspection (-1: absorbed or after the end)
    t = np.zeros(l); state = np.zeros(l, dtype=np.int64); alive = np.arange(l)
    while alive.size:
        st = state[alive]
        t1 = t[alive] + rng.exponential(1.0, alive.size) / rate[st]
        inside = (ins[None, :] >= t[alive][:, None]) & (ins[None, :] < t1[:, None])
        rows, cols = np.nonzero(inside)
        seen[alive[rows], cols] = st[rows]
        t[alive] = t1
        nxt = (rng.random(alive.size)[:, None] >= cum[st]).sum(1)
        state[alive] = nxt
        alive = alive[nxt < n]
    cens = t > end
    y = np.where(cens, end, t)
    keep = (seen >= 0) & (ins[None, :] <= y[:, None])
    counts = keep.sum(1)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    rows, cols = np.nonzero(keep)
    return y, cens.astype(np.int32), offsets, ins[cols], masks[stage[seen[rows, cols]]]


def misclassified_panel(R, s, l, spacing, k, E, rng, censor=None):
    """Misclassified panel data (Engine.set_stage_visits): panel(R, s, l, spacing, k, ...) with every phase seen exactly,
    then each visit's stage read from row c of the emission matrix E (n, S) for the true phase c.  Returns (y, censored,
    offsets, t, stage, phase), phase the true phase at each visit."""
    n = s.shape[0]
    E = np.asarray(E, dtype=np.float64)
    y, cens, offsets, t, mask = panel(R, s, l, spacing, k, np.arange(n), rng, censor=censor)
    phase = np.log2(mask.astype(np.float64)).astype(np.int64)
    cum = np.cumsum(E, axis=1)
    cum[:, -1] = 1.0
    stage = (rng.random(phase.size)[:, None] >= cum[phase]).sum(1)
    return y, cens, offsets, t, stage.astype(np.uint32), phase


def tabulate(y, cens, u=None):
    """Tied observations as records with counts (Engine.set_counts): the distinct (y, cens, u) in order of first occurrence
    and how often each occurs.  Returns (y, cens, u, counts) with u None when no u was given; np.repeat of the records by
    the counts gives back the observations, grouped by record."""
    y = np.asarray(y, dtype=np.float64); c = np.asarray(cens, dtype=np.int32)
    cols = [y.view(np.uint64), c.astype(np.uint64)]
    if u is not None:
        cols.append(np.asarray(u, dtype=np.float64).view(np.uint64))
    _, first, counts = np.unique(np.stack(cols, axis=1), axis=0, return_index=True, return_counts=True)
    order = np.argsort(first, kind="stable")
    idx = first[order]
    return (y[idx], c[idx], None if u is None else np.asarray(u, dtype=np.float64)[idx], counts[order].astype(np.uint32))


def delayed_entry(R, s, l, entry, rng, censor=None, spacing=None):
    """Delayed-entry (left-truncated) data: l units of the CTMC (R, s) started in state 0 that were still working at their
    entry ages.  entry(k, rng) draws k candidate ages; a unit absorbed at or before its age never enters the sample and is
    redrawn.  censor(k, rng), when given, draws k study-end ages: a unit still working then is right-censored there
    (units whose study ends at or before entry are redrawn too).  With spacing the units are inspected every spacing time
    units from entry on, and a unit found failed gives the interval y = a + (i-1) spacing, u = a + i spacing.
    Returns (y, a): exact failure times and entry ages; with censor or spacing (y, a, censored, u), u = +inf where there
    is no upper bound."""
    ys, As, cs, us = [], [], [], []
    need = l
    while need > 0:
        k = max(2 * need, 1024)
        t = simulate_pht(R, s, k, rng)
        a = np.asarray(entry(k, rng), dtype=np.float64)
        end = np.full(k, np.inf) if censor is None else np.asarray(censor(k, rng), dtype=np.float64)
        keep = (t > a) & (end > a)
        t, a, end = t[keep][:need], a[keep][:need], end[keep][:need]
        cens = t > end
        y = np.where(cens, end, t)
        u = np.full(y.shape[0], np.inf)
        if spacing is not None:
            i = np.ceil((y - a) / spacing)
            fail = ~cens
            y = np.where(fail, a + (i - 1) * spacing, y)
            u = np.where(fail, a + i * spacing, u)
            cens = np.ones(y.shape[0], dtype=bool)
        ys.append(y); As.append(a); cs.append(cens.astype(np.int32)); us.append(u)
        need -= y.shape[0]
    if censor is None and spacing is None:
        return np.concatenate(ys), np.concatenate(As)
    return np.concatenate(ys), np.concatenate(As), np.concatenate(cs), np.concatenate(us)


def structure_rates(T, C, theta, n):
    """(R, s) of the generator that theta maps to through the structure (T, C): column-major flat (n+1)^2, as pht_config
    takes them."""
    T = np.asarray(T).reshape(n + 1, n + 1, order="F"); C = np.asarray(C, dtype=np.float64).reshape(n + 1, n + 1, order="F")
    rate = np.where(T > 0, np.asarray(theta, dtype=np.float64)[np.maximum(T, 1) - 1] * C, 0.0)
    R = rate[:n, :n].copy(); np.fill_diagonal(R, 0.0)
    return R, rate[:n, n].copy()


def groups(T, C, theta, n, sizes, rng, censor=None):
    """Grouped data (Engine.set_groups): G structures T[g], C[g] (column-major flat (n+1)^2 each) over one parameter vector
    theta.  Group g gets sizes[g] absorption times of its own generator (structure_rates), started in state 0
    (simulate_pht).  censor(k, rng), when given, draws k censoring times: a unit still working then is right-censored
    there.  Returns (y, censored, group), the groups one after another."""
    ys, cs, gs = [], [], []
    for g, k in enumerate(sizes):
        R, s = structure_rates(T[g], C[g], theta, n)
        t = simulate_pht(R, s, int(k), rng)
        end = np.full(int(k), np.inf) if censor is None else np.asarray(censor(int(k), rng), dtype=np.float64)
        ys.append(np.minimum(t, end)); cs.append((t > end).astype(np.int32)); gs.append(np.full(int(k), g, dtype=np.int32))
    return np.concatenate(ys), np.concatenate(cs), np.concatenate(gs)


def _general_T(R, s):
    """Every non-zero rate its own parameter, numbered column-major like sorted "Sij"/"si" names would be."""
    n = s.shape[0]
    T = np.zeros((n + 1, n + 1), dtype=np.int32)
    theta = []
    for j in range(n + 1):
        for i in range(n):
            v = s[i] if j == n else R[i, j]
            if i != j and v != 0.0:
                theta.append(v); T[i, j] = len(theta)
    return T, np.ones((n + 1, n + 1)), np.array(theta)


def _finish(name, R, s, T, C, theta, l, frac_cens, rng, shard=None):
    if shard is not None:           # weak-scaling runs: same model, an independent data stream per shard
        rng = np.random.default_rng([SEED0, 0x5348, int(shard)])
    y = simulate_pht(R, s, l, rng)
    cens = np.zeros(l, dtype=np.int32)
    if frac_cens > 0:
        flag = rng.random(l) < frac_cens
        y = np.where(flag, y * rng.random(l), y)          # censoring time = U(0,1) x true time
        y = np.maximum(y, 1e-12)
        cens = flag.astype(np.int32)
    nu = np.full(theta.shape[0], 2.0)
    zeta = 2.0 / theta
    return Workload(name, s.shape[0], T.ravel(order="F").copy(), C.ravel(order="F").copy(), theta, nu, zeta, y, cens, R, s)


def dense(n, l, frac_cens, symmetric, seed, name, shard=None):
    rng = np.random.default_rng(seed)
    R = rng.uniform(0.2, 1.2, (n, n))
    if symmetric:
        R = (R + R.T) / 2
    np.fill_diagonal(R, 0.0)
    s = rng.uniform(0.2, 1.2, n)
    T, C, theta = _general_T(R, s)
    return _finish(name, R, s, T, C, theta, l, frac_cens, rng, shard)


def config(cid, method="MHRS", l=None, shard=None):
    """Workload of BASELINE.json configs[cid-1] (cid = 1..5); l overrides the observation count; shard = k gives the
    k-th independent data set of the same model (rank k of a weak-scaling run)."""
    sym = method in ("ECS", "DCS")
    if cid == 1:
        S = np.array([[-3.6, 1.8, 1.8], [9.5, -11.3, 0.0], [9.5, 0.0, -11.3]])
        R = S.copy(); np.fill_diagonal(R, 0.0)
        s = -S.sum(1)
        T, C, theta = _general_T(R, s)
        return _finish("C1: 3-phase package example", R, s, T, C, theta, l or 100, 0.0, np.random.default_rng(SEED0 + 1), shard)
    if cid == 2:
        n = 4
        R = np.zeros((n, n)); s = np.full(n, 0.3)
        for i in range(n - 1):
            R[i, i + 1] = 1.0 + 0.37 * i
        s[n - 1] = 1.5
        T, C, theta = _general_T(R, s)
        return _finish("C2: 4-phase Coxian, exact", R, s, T, C, theta, l or 10 ** 6, 0.0, np.random.default_rng(SEED0 + 2), shard)
    if cid == 3:
        return dense(8, l or 10 ** 7, 0.2, sym, SEED0 + 3, "C3: 8-phase dense%s, 20%% right-censored" % (" symmetric" if sym else ""), shard)
    if cid == 5:
        return dense(32, l or 10 ** 8, 0.0, sym, SEED0 + 5, "C5: 32-phase dense%s" % (" symmetric" if sym else ""), shard)
    if cid == 4:
        return series_parallel(l or 10 ** 7, shard=shard)
    raise ValueError("config id must be 1..5")


def series_parallel(l, seed=SEED0 + 4, f=0.5, r=4.0, shard=None):
    """C4: two 2-out-of-3 blocks in series (6 independent repairable components): the system is up while
    each block has at most one failed component, which gives 4 x 4 = 16 up-states = the transient phases.
    Every failure cell is the tied parameter F and every repair cell R (the structure of
    tests/phtMCMC2.R:15 scaled up); failures that take the system down go to the absorbing column with
    their multiplicity in C.  Start: all components up."""
    comps = 6
    states = [tuple((k >> c) & 1 for c in range(comps)) for k in range(1 << comps)]      # 1 = failed

    def up(st):
        return (st[0] + st[1] + st[2]) <= 1 and (st[3] + st[4] + st[5]) <= 1
    ups = [st for st in states if up(st)]
    ups.sort(key=lambda st: (sum(st), st))
    idx = {st: k for k, st in enumerate(ups)}
    n = len(ups)
    T = np.zeros((n + 1, n + 1), dtype=np.int32); C = np.ones((n + 1, n + 1))
    R = np.zeros((n, n)); s = np.zeros(n)
    F_ID, R_ID = 1, 2                                   # sorted names: "F" < "R"
    for st in ups:
        i = idx[st]
        for c in range(comps):
            nxt = list(st); nxt[c] ^= 1; nxt = tuple(nxt)
            if st[c] == 0:                              # failure of component c
                if up(nxt):
                    T[i, idx[nxt]] = F_ID; R[i, idx[nxt]] = f
                else:                                   # system failure: absorbing column, multiplicity through C
                    if T[i, n] == 0:
                        T[i, n] = F_ID; C[i, n] = 0.0
                    C[i, n] += 1.0; s[i] += f
            else:                                       # repair of component c
                T[i, idx[nxt]] = R_ID; R[i, idx[nxt]] = r
    theta = np.array([f, r])
    rng = np.random.default_rng(seed)
    return _finish("C4: 16-state series-parallel, tied F/R", R, s, T, C, theta, l, 0.0, rng, shard)
