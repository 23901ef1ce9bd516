"""Instruction count of the MHRS filter jump-step in the SASS of the search kernels, by pipe class.

    python tools/sass_step_count.py [--obj k_mhrs.cu.o] [--src k_mhrs.cu] [--nc 8]

Builds phasetype_b200/csrc/k_mhrs.cu for sm_100a with the flags of phasetype_b200/build.py (or reads an object built
already, --obj) and reads `cuobjdump -sass` of k_mhrs_lanes<NC, IV> and k_mhrs_tail<NC, IV>.  Needs nvcc and cuobjdump,
no GPU.

The step loop of a kernel is the innermost loop (a backward branch and its target) that contains the step's MUFU.LG2;
a loop body that runs several jump-steps per trip holds one MUFU.LG2 for each.  Counts are static: every instruction
of the loop once, per jump-step (divided by the steps per trip).  `rare` is the part inside nested loops that hold no
MUFU.LG2 (the threshold scan of a guide bucket with a threshold in it, about 1 look-up in 25 at 8 phases); `common` is
the rest.  In the tail kernel the loop also holds the pool hand-out code, which runs when a pool is used up.

Pipe classes, by opcode (a reading of the public opcode tables, not a hardware measurement):
  ALU      integer logic, compares, selects, shifts, byte permutes, votes, popc, integer adds that are not IMAD
  FMA      FFMA / FADD / FMUL and every IMAD form (IMAD.MOV and IMAD.IADD included: ptxas uses them to move work off ALU)
  FP64     DFMA / DADD / DMUL / DSETP
  XU       MUFU and the conversions that go through it
  LSU      shared, global and local memory, shuffles, atomics (LDL / STL are also listed on their own)
  uniform  the uniform datapath (U*, LDCU, R2UR, S2UR, VOTEU)
  other    branches, convergence barriers, S2R, LDC, NOP
"""
import argparse
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ALU = {"LOP3", "LOP", "ISETP", "FSETP", "SEL", "FSEL", "PRMT", "LEA", "SHF", "SHL", "SHR", "PLOP3", "POPC", "VOTE",
       "IADD3", "IADD", "MOV", "VIADD", "VIMNMX", "IMNMX", "FMNMX", "IABS", "P2R", "R2P", "BMSK", "SGXT", "FLO", "BREV",
       "I2FP", "F2FP", "FCHK", "ISCADD", "LEPC"}
FMA = {"FFMA", "FADD", "FMUL", "IMAD", "IMUL", "FSWZADD", "IDP"}
FP64 = {"DFMA", "DADD", "DMUL", "DSETP", "DMNMX"}
XU = {"MUFU", "I2F", "F2I", "F2F", "FRND"}
LSU = {"LDS", "STS", "LDG", "STG", "LDL", "STL", "LD", "ST", "ATOMS", "ATOMG", "ATOM", "RED", "REDG", "SHFL", "LDSM",
       "MATCH", "LDGSTS"}
CLASSES = ("ALU", "FMA", "FP64", "XU", "LSU", "uniform", "other")


def pipe_of(op):
    base = op.split(".")[0]
    if base in ("LDCU", "R2UR", "S2UR", "VOTEU") or base.startswith("U"):
        return "uniform"
    for name, ops in (("ALU", ALU), ("FMA", FMA), ("FP64", FP64), ("XU", XU), ("LSU", LSU)):
        if base in ops:
            return name
    return "other"


LINE = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)\s*([^;]*);")


def parse(sass):
    ins = []
    for m in LINE.finditer(sass):
        ins.append((int(m.group(1), 16), m.group(3), m.group(4).strip()))
    return ins


def loops(ins):
    """(start, end) address ranges of backward branches, end = the branch itself"""
    out = []
    for addr, op, args in ins:
        if op.split(".")[0] in ("BRA", "JMP"):
            m = re.search(r"0x([0-9a-f]+)\s*$", args)
            if m and int(m.group(1), 16) <= addr:
                out.append((int(m.group(1), 16), addr))
    return out


def step_loop(ins):
    lg2 = [a for a, op, _ in ins if op.startswith("MUFU.LG2")]
    cands = [(s, e) for s, e in loops(ins) if any(s <= a <= e for a in lg2)]
    if not cands:
        raise SystemExit("no loop with a MUFU.LG2 found")
    s, e = min(cands, key=lambda r: r[1] - r[0])
    steps = sum(1 for a in lg2 if s <= a <= e)
    inner = [(s2, e2) for s2, e2 in loops(ins) if s < s2 <= e2 < e and not any(s2 <= a <= e2 for a in lg2)]
    return s, e, steps, inner


def count(ins, s, e, inner):
    tot = {c: 0 for c in CLASSES + ("rare", "local")}
    for addr, op, _ in ins:
        if not (s <= addr <= e):
            continue
        if any(s2 <= addr <= e2 for s2, e2 in inner):
            tot["rare"] += 1
            continue
        tot[pipe_of(op)] += 1
        if op.startswith(("LDL", "STL")):
            tot["local"] += 1
    return tot


def build_obj(src, out):
    from phasetype_b200 import build as b
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    subprocess.run([nvcc] + b.NVCC_FLAGS + ["-I", os.path.dirname(os.path.abspath(src)), "-c", src, "-o", out], check=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--obj", help="a k_mhrs.cu object built already (default: build --src)")
    ap.add_argument("--src", default=os.path.join(ROOT, "phasetype_b200", "csrc", "k_mhrs.cu"))
    ap.add_argument("--nc", type=int, default=8, choices=(8, 16, 32))
    a = ap.parse_args()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    with tempfile.TemporaryDirectory() as tmp:
        obj = a.obj
        if obj is None:
            obj = os.path.join(tmp, "k_mhrs.o")
            build_obj(a.src, obj)
        hdr = "%-22s %5s %6s " % ("kernel", "steps", "total") + " ".join("%7s" % c for c in CLASSES) + " %6s %6s" % ("rare", "local")
        print(hdr)
        for kern, mangled in (("lanes", "_Z12k_mhrs_lanesILi%dELb%dEEv11SweepParams"), ("tail", "_Z11k_mhrs_tailILi%dELb%dEEv11SweepParams")):
            for iv in (0, 1):
                name = mangled % (a.nc, iv)
                sass = subprocess.run([cuobjdump, "-sass", "-fun", name, obj], check=True, capture_output=True, text=True).stdout
                ins = parse(sass)
                s, e, steps, inner = step_loop(ins)
                t = count(ins, s, e, inner)
                common = sum(t[c] for c in CLASSES)
                print("%-22s %5d %6.1f " % ("%s<%d,%s>" % (kern, a.nc, "true" if iv else "false"), steps, common / steps)
                      + " ".join("%7.1f" % (t[c] / steps) for c in CLASSES) + " %6.1f %6d" % (t["rare"] / steps, t["local"]))


if __name__ == "__main__":
    main()
