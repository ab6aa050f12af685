#!/usr/bin/env python
"""Static SASS of the funnel's rn_k_iter for a set of RN_X_* switches (no device): instruction count, opcode mix, branches,
registers, of the whole kernel and of the leapfrog loop (between the two backward branches with the largest span).
Usage: python scripts/r2b/sass_iter.py "<defs A>" "<defs B>" ...   (RN_MAXRREGCOUNT from the environment)"""
import collections, os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from rainier_b200 import api

rir = open(os.path.join(ROOT, "rainier_b200", "models", "funnel10.rir"), "rb").read()
cfg = api.make_config(iterations=100, warmupIterations=0, sampler=api.HMCSampler(5), stepSizeTuner=api.StaticStepSize(0.1),
                      massMatrixTuner=api.IdentityMassMatrixTuner(), launchIterations=100)
for defs in (sys.argv[1:] or [""]):
    m = api.CudaModel(rir, [], device=-1)
    cub = "/tmp/sass_iter.cubin"
    open(cub, "wb").write(m.emit_cubin(cfg))
    m.close()
    res = subprocess.run(["cuobjdump", "-res-usage", cub], capture_output=True, text=True).stdout
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", "rn_k_iter", cub], capture_output=True, text=True).stdout
    ins = []
    for l in sass.splitlines():
        mm = re.match(r"\s+/\*([0-9a-f]+)\*/\s+(.*?);", l)
        if mm:
            ins.append((int(mm.group(1), 16), re.sub(r"^@!?U?P\d+\s+", "", mm.group(2).strip())))
    regs = re.search(r"Function rn_k_iter:\s*\n?\s*REG:(\d+) STACK:(\d+)", res)
    c = collections.Counter(t.split()[0].split(".")[0] for _, t in ins)
    ctl = sum(c[k] for k in ("BRA", "BSSY", "BSYNC", "CALL", "RET", "BREAK", "WARPSYNC"))
    fp = sum(c[k] for k in ("DADD", "DMUL", "DFMA", "DSETP"))
    print("defs=%r regs/stack=%s total=%d fp64=%d control=%d IMAD=%d UMOV=%d MUFU=%d CALL=%d" % (
        defs, regs.groups() if regs else None, len(ins), fp, ctl, c["IMAD"], c["UMOV"], c["MUFU"], c["CALL"]))
    # loops: backward branches
    loops = []
    for a, t in ins:
        mm = re.match(r"BRA(?:\.\w+)* (?:\w+, )?0x([0-9a-f]+)", t)
        if mm and int(mm.group(1), 16) <= a:
            loops.append((int(mm.group(1), 16), a))
    for lo, hi in sorted(loops, key=lambda x: x[0] - x[1])[:4]:
        body = [t for a, t in ins if lo <= a <= hi]
        cc = collections.Counter(t.split()[0].split(".")[0] for t in body)
        print("   loop 0x%x..0x%x: %d instr, fp64 %d, BRA %d, BSSY %d, CALL %d, MUFU %d" % (
            lo, hi, len(body), sum(cc[k] for k in ("DADD", "DMUL", "DFMA", "DSETP")), cc["BRA"], cc["BSSY"], cc["CALL"], cc["MUFU"]))
