"""Drop-in boundary checks that need no GPU: the shared library loads, exports every symbol include/pht_b200.h
declares, refuses to run without a CUDA device (no CPU fallback), and the Python mirrors of the R wrappers
validate their arguments like the R code does."""
import os
import re
import subprocess

import numpy as np
import pytest

import phasetype_b200 as pb
from phasetype_b200 import _lib, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "pht_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(LJMA_Gibbs|pht_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from phasetype_b200 import build
    build.build()
    names = header_functions()
    assert "LJMA_Gibbs" in names and len(names) >= 18
    assert sorted(_lib.SYMBOLS) == names
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if line.strip()}
    for nm in names:
        assert nm in exported, nm
    L = pb.lib()
    for nm in names:
        assert hasattr(L, nm)


def test_ljma_gibbs_signature_is_the_registered_one():
    """15 pointer arguments in the order of reference src/PHT_MCMC_Aslett.h:1-3 / src/Registrations.c:6-12."""
    src = open(os.path.join(ROOT, "include", "pht_b200.h")).read()
    m = re.search(r"void LJMA_Gibbs\((.*?)\);", src, flags=re.S)
    args = [a.strip() for a in m.group(1).replace("\n", " ").split(",")]
    assert [a.split("*")[-1].strip() for a in args] == ["it", "mhit", "method", "n", "m", "nu", "zeta", "T", "C", "y", "l",
                                                        "censored", "start", "silent", "res"]
    assert [a.split("*")[0].strip() for a in args] == ["int"] * 5 + ["double"] * 2 + ["int"] + ["double"] * 2 + ["int"] * 2 + \
        ["double", "int", "double"]


@pytest.mark.skipif(pb.lib().pht_device_count() > 0, reason="a GPU is present")
def test_no_cpu_fallback():
    with pytest.raises(pb.EngineError, match="no CUDA device"):
        pb.Engine(3, np.zeros(16, dtype=np.int32), np.ones(16), [1.0], [1.0], [1.0], [0], method=1)
    os.environ["PHT_B200_QUIET"] = "1"
    res = pb.ljma_gibbs(5, 1, 1, 3, 2, [24, 180], [16, 16], [0, 2, 2, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 1, 1, 0], np.ones(16),
                        [1.0, 2.0], [0, 0], [-1.0])
    assert np.allclose(res[0], [23 / 16, 179 / 16])       # start row = prior mode (src/PHT_MCMC_Aslett.c:197-198)
    assert np.isnan(res[1:]).all()                         # nothing was computed on the CPU: the rows are NA, not zeros
    with pytest.raises(pb.EngineError):
        pb.fp64_fma_rate()


def test_zbits_rule():
    L = pb.lib()
    assert L.pht_choose_zbits(1.0) == 52 and L.pht_choose_zbits(1e7) == 34 and L.pht_choose_zbits(1e9) == 28    # capped at 52 bits
    from oracle import pyoracle as po
    for v in (1e-3, 1.0, 123.4, 1e7, 3e9):
        assert L.pht_choose_zbits(v) == po.choose_zbits(v)


def test_wrapper_argument_checks_follow_the_r_code():
    x = [1.0, 2.0]
    TT = np.array([["0", "F", "F", "0"], ["R", "0", "0", "F"], ["R", "0", "0", "F"], ["0", "0", "0", "0"]], dtype=object)
    nu = {"R": 180, "F": 24}; zeta = {"R": 16, "F": 16}
    with pytest.raises(ValueError, match="invalid number of MCMC iterations"):
        api.phtMCMC2(x, TT, [1, 0, 0], nu, zeta, 0)
    with pytest.raises(ValueError, match="must be square"):
        api.phtMCMC2(x, TT[:3], [1, 0, 0], nu, zeta, 5)
    bad = TT.copy(); bad[1, 1] = "R"
    with pytest.raises(ValueError, match="diagonal"):
        api.phtMCMC2(x, bad, [1, 0, 0], nu, zeta, 5)
    bad = TT.copy(); bad[3, 0] = "R"
    with pytest.raises(ValueError, match="last row"):
        api.phtMCMC2(x, bad, [1, 0, 0], nu, zeta, 5)
    with pytest.raises(ValueError, match="beta should be a vector of length 3"):
        api.phtMCMC2(x, TT, [1, 0], nu, zeta, 5)
    with pytest.raises(ValueError, match="don't match those in prior nu"):
        api.phtMCMC2(x, TT, [1, 0, 0], {"R": 1}, zeta, 5)
    with pytest.raises(ValueError, match="unknown sampling methods"):
        api.phtMCMC2(x, TT, [1, 0, 0], nu, zeta, 5, method="HMC")
    names, TN = api._encode(TT, nu, zeta)
    assert names == ["F", "R"]
    assert TN.ravel(order="F").tolist() == [0, 2, 2, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 1, 1, 0]      # SURVEY Appendix C, fixture 2
    with pytest.raises(ValueError, match="nu must specify"):
        api.phtMCMC(x, 3, [1, 0, 0], [1.0] * 8, [1.0] * 3, 5)
    with pytest.raises(ValueError):                      # 11 states: "S111" names collide, as upstream (R/phtMCMC.R:17)
        api.phtMCMC(x, 11, np.ones(11), np.ones(121), np.ones(11), 5)


@pytest.mark.parametrize("kw,msg", [(dict(n=0), "outside 1.."), (dict(n=33), "outside 1.."), (dict(method=32), "unknown sampling method"),
                                    (dict(mhit=-1), "mhit"), (dict(rank=2, world=2), "bad shard"), (dict(zbits=60), "zbits")])
def test_engine_rejects_bad_arguments_before_touching_the_device(kw, msg):
    a = dict(n=3, method=1, mhit=1, rank=0, world=1, zbits=30); a.update(kw)
    n1 = max(a["n"], 1) + 1
    with pytest.raises(pb.EngineError, match=msg):
        pb.Engine(a["n"], np.zeros(n1 * n1, dtype=np.int32), np.ones(n1 * n1), [1.0], [1.0], [1.0], [0], method=a["method"],
                  mhit=a["mhit"], rank=a["rank"], world=a["world"], zbits=a["zbits"])


def test_several_ranks_need_a_common_fixed_point_scale():
    """A per-rank guess of zbits from the local sum of y can differ between ranks near a power of two (ADVICE round 1)."""
    with pytest.raises(pb.EngineError, match="several ranks"):
        pb.Engine(3, np.zeros(16, dtype=np.int32), np.ones(16), [1.0], [1.0], [1.0], [0], method=1, rank=0, world=2)


def test_weak_scaling_shards_share_the_model():
    from phasetype_b200 import synth
    a = synth.config(3, "MHRS", l=500); b = synth.config(3, "MHRS", l=500, shard=1); c = synth.config(3, "MHRS", l=500, shard=1)
    assert np.array_equal(a.theta, b.theta) and np.array_equal(a.T, b.T)
    assert not np.array_equal(a.y, b.y) and np.array_equal(b.y, c.y)


def test_product_path_never_touches_the_checker():
    """oracle/ is test infrastructure: nothing under phasetype_b200/ or include/ may import, include or link it, and
    bench.py may only reach it from the CPU-baseline / reference-arm legs."""
    import ast
    bad = []
    for base in ("phasetype_b200", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            if os.path.basename(dirpath) in ("build", "__pycache__"):
                continue
            for f in files:
                if not f.endswith((".py", ".c", ".h", ".cu", ".cuh")):
                    continue
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                if re.search(r'#\s*include\s*["<][^">]*oracle|(from|import)\s+oracle|pyoracle|libphtoracle|libphtref|\bpho_[a-z_]+\s*\(', txt):
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad
    tree = ast.parse(open(os.path.join(ROOT, "bench.py")).read())
    allowed = {"_cpu_worker", "ref_kind", "main"}         # main: only inside the `cpu_baseline` block, checked below
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef):
            for sub in ast.walk(node):
                if isinstance(sub, ast.ImportFrom) and sub.module == "oracle":
                    assert node.name in allowed, node.name
    src = open(os.path.join(ROOT, "bench.py")).read()
    main_src = src[src.index("def main():"):]
    assert main_src.count("from oracle import") == 1 and "if not args.no_cpu:" in main_src.split("from oracle import")[0][-400:]


@pytest.mark.skipif(pb.lib().pht_device_count() > 0, reason="a GPU is present")
def test_start_row_follows_the_reference_rule_without_a_device():
    """Row 0 of res is produced by the host routine before any device work: prior mode (nu - 1) / zeta where nu > 1, a
    prior draw from the keyed parameter stream otherwise (src/PHT_MCMC_Aslett.c:195-207) -- the same numbers as the
    checker's driver; user-supplied start values are copied through."""
    from oracle import pyoracle as po
    os.environ["PHT_B200_SEED"] = "4242"; os.environ["PHT_B200_QUIET"] = "1"
    T = [0, 2, 2, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 1, 1, 0]; Cm = np.ones(16)
    y = np.array([1.0, 2.0, 0.5]); cens = np.zeros(3, dtype=np.int32)
    nu = [0.7, 180.0]; zeta = [16.0, 16.0]
    res = pb.ljma_gibbs(3, 1, 2, 3, 2, nu, zeta, T, Cm, y, cens, [-1.0])
    want, _ = po.gibbs(4242, 3, 1, 2, 3, nu, zeta, T, Cm, y, cens, [-1.0])
    assert res[0, 1] == 179.0 / 16.0 and res[0, 0] > 0
    assert np.array_equal(res[0], want[0])
    res = pb.ljma_gibbs(3, 1, 2, 3, 2, nu, zeta, T, Cm, y, cens, [0.25, 7.5])
    assert np.array_equal(res[0], [0.25, 7.5]) and np.isnan(res[1:]).all()


def test_reference_registration_table_binds_the_drop_in():
    """The reference's src/Registrations.c, unmodified, compiled against stand-in R headers and linked with
    libpht_b200.so (oracle/Makefile `reg`): R_init_PhaseType must register LJMA_Gibbs as a 15-argument .C routine with
    the reference's argument types, pointing at the product library's symbol, and switch dynamic lookup off."""
    import ctypes as C
    from oracle import pyoracle as po
    if not os.path.exists(po.REG_SO):
        pytest.skip("oracle/_ref/PhaseType_reg.so not built (needs PHT_REFERENCE_SRC)")
    reg = C.CDLL(po.REG_SO)
    fun = C.c_void_p(); nargs = C.c_int(); types = (C.c_uint * 32)(); dyn = C.c_int(); force = C.c_int()
    assert reg.phtreg_lookup(b"LJMA_Gibbs", C.byref(fun), C.byref(nargs), types, 32, C.byref(dyn), C.byref(force)) == 0
    INT, REAL = 13, 14
    assert nargs.value == 15
    assert list(types[:15]) == [INT] * 5 + [REAL] * 2 + [INT] + [REAL] * 2 + [INT] * 2 + [REAL, INT, REAL]
    assert dyn.value == 0 and force.value == 1
    assert fun.value == C.cast(pb.lib().LJMA_Gibbs, C.c_void_p).value
    assert hasattr(reg, "R_init_PhaseType")
