#!/usr/bin/env python
"""Writes profiles/<tag>_sass_excerpts.txt: mnemonic counts of every kernel of the shipped library and the hot loops of the
three hot kernels (blend hit evaluation, onesweep ranking, fused preprocess SH staging), from `cuobjdump -sass`.

    python scripts/sass_excerpt.py r02
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "luisacomputegaussiansplatting_b200", "liblcgs_b200.so")
tag = sys.argv[1] if len(sys.argv) > 1 else "rXX"

sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
funcs, name = collections.OrderedDict(), None
for ln in sass.splitlines():
    m = re.search(r"Function : (\S+)", ln)
    if m:
        name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
        name = re.sub(r"\(.*", "", name)
        funcs[name] = []
    elif name and re.match(r"\s+/\*[0-9a-f]{4}\*/", ln):
        funcs[name].append(re.sub(r"\s*/\* 0x[0-9a-f]+ \*/\s*$", "", ln).rstrip())

arch = re.findall(r"arch = (sm_\w+)", sass)
out = ["SASS of %s (cuobjdump -sass), architectures: %s" % (os.path.relpath(LIB, ROOT), sorted(set(arch))), ""]
keys = ["LDG", "STG", "LDS", "STS", "LDGSTS", "ATOMS", "ATOMG", "RED", "BAR", "VOTE", "MATCH", "SHFL", "MUFU.EX2", "MUFU", "FFMA", "FMUL",
        "FADD", "FFMA2", "FMUL2", "FADD2", "DFMA", "DMUL", "FLO", "UBLKCP", "UTMALDG", "UTCMMA", "HMMA", "STL", "LDL"]
out.append("%-78s %5s  %s" % ("kernel", "instr", "mnemonic counts (static)"))
for f, lines in funcs.items():
    ops = collections.Counter()
    for ln in lines:
        m = re.search(r"\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", ln)
        if m:
            op = m.group(1)
            for k in keys:
                if op == k or op.startswith(k + "."):
                    ops[k] += 1
    out.append("%-78s %5d  %s" % (f[:78], len(lines), " ".join("%s=%d" % (k, ops[k]) for k in keys if ops[k])))
out.append("")
out.append("No UTCMMA / HMMA (no stage is a dense contraction) and no UBLKCP / UTMALDG (TMA staging was measured slower than")
out.append("register prefetch + LDGSTS, profiles/README.md); STL / LDL = local-memory spills.")


def excerpt(title, fname_part, start_pat, end_pat, before=0, after=0):
    for f, lines in funcs.items():
        if fname_part in f:
            idx = [i for i, ln in enumerate(lines) if re.search(start_pat, ln)]
            if not idx:
                continue
            a = max(0, idx[0] - before)
            b = next((i for i in range(idx[0], len(lines)) if re.search(end_pat, lines[i])), min(len(lines) - 1, idx[0] + 60))
            out.append("")
            out.append("---- %s ----" % title)
            out.append("     %s, instructions %d..%d of %d" % (f, a, b + after, len(lines)))
            out.extend(lines[a:b + after + 1])
            return


excerpt("blend: the hit-evaluation loop (one (Gaussian, 8x8 patch) pair per iteration, two pixels per lane: FLO / BMSK walk of the ballot, "
        "three broadcast LDS.128, power on FADD2 / FMUL2 / FFMA2, threshold compares, 2 x MUFU.EX2, blend)", "blend2_kernel<10>", r"FLO\.U32", r"@P\d BRA", before=1, after=0)
excerpt("onesweep<u64, 256x20, 7-bit digits, HI>: ranking of one item (7 x [LOP3 test, VOTE, SEL, LOP3], ATOMS by the group leader, SHFL)",
        "onesweep_pass_kernel<unsigned long long, 256, 20, 7, 2, false, true>", r"VOTE\.ANY", r"SHFL\.IDX", before=2, after=2)
excerpt("onesweep<u64, 256x20>: the scatter -- keys by STS.64, values by LDGSTS (global -> shared, no register)",
        "onesweep_pass_kernel<unsigned long long, 256, 20, 7, 2, false, true>", r"LDGSTS", r"LDGSTS.*\n|BAR", before=6, after=8)
excerpt("preprocess_fused<true>: predicated, coalesced SH staging with LDGSTS.128", "preprocess_fused_kernel<true>", r"LDGSTS", r"LDGDEPBAR|DEPBAR",
        before=3, after=1)
path = os.path.join(ROOT, "profiles", "%s_sass_excerpts.txt" % tag)
open(path, "w").write("\n".join(out) + "\n")
print(path, len(out), "lines")
