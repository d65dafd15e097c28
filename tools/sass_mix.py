"""Instruction mix of every kernel in liblrb200.so from `cuobjdump -sass` (runs without a GPU).

    python tools/sass_mix.py [lrbinner_b200/liblrb200.so] > profiles/rNN_sass_mix.csv

One row per kernel instantiation: static instruction counts by class.  The columns that matter for this path:
LDG/STG (global), LDS/STS/ATOMS (shared), RED/ATOMG (global atomics), MATCH/SHFL/VOTE (warp aggregation),
SHF/LOP3/IADD (the key arithmetic), BAR, LDS.128/STG.128 (16-byte accesses, also counted in LDS/STG), and the Blackwell data-movement mnemonics (UBLKCP = cp.async.bulk,
UTMALDG/UTMASTG = TMA tensor copies, LDGSTS = cp.async, SYNCS = mbarrier) so that their presence or absence is on record.
"""
import collections
import re
import subprocess
import sys

CLASSES = [("LDG", r"^LDG"), ("STG", r"^STG"), ("LDS", r"^LDS"), ("STS", r"^STS"), ("ATOMS", r"^ATOMS"), ("RED", r"^RED"),
           ("ATOMG", r"^ATOMG|^ATOM\b"), ("LDC", r"^LDC|^ULDC|^LDCU"), ("MATCH", r"^MATCH"), ("SHFL", r"^SHFL"), ("VOTE", r"^VOTE"),
           ("SHF", r"^SHF"), ("LOP3", r"^LOP3|^ULOP3"), ("IADD", r"^IADD|^UIADD|^IMAD|^LEA"), ("ISETP", r"^ISETP|^UISETP"), ("SEL", r"^SEL|^USEL"),
           ("POPC/BREV/FLO", r"^POPC|^BREV|^FLO"), ("BAR", r"^BAR"), ("BRA", r"^BRA|^BSSY|^BSYNC|^EXIT"),
           ("UBLKCP", r"^UBLKCP"), ("UTMA", r"^UTMALDG|^UTMASTG|^UTMAPF"), ("LDGSTS", r"^LDGSTS"), ("SYNCS", r"^SYNCS"), ("TCGEN05", r"^UTC|^TCGEN")]
# 16-byte accesses, counted a second time beside their class (LDS / STG)
WIDE = [("LDS.128", r"^LDS\.128"), ("STG.128", r"^STG(\.E)?\.128")]


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    res = []
    for s in out:
        s = re.sub(r"\(anonymous namespace\)::", "", s)
        s = re.sub(r"^void ", "", s)
        res.append(s.split("(")[0])
    return res


def main(path="lrbinner_b200/liblrb200.so"):
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True).stdout
    funcs, cur = collections.OrderedDict(), None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = collections.Counter()
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m and cur:
            op = m.group(1)
            funcs[cur]["total"] += 1
            for name, pat in CLASSES:
                if re.match(pat, op):
                    funcs[cur][name] += 1
                    break
            for name, pat in WIDE:
                if re.match(pat, op):
                    funcs[cur][name] += 1
    names = demangle(list(funcs))
    cols = ["total"] + [c for c, _ in CLASSES] + [c for c, _ in WIDE]
    print("kernel," + ",".join(cols))
    for nm, cnt in sorted(zip(names, funcs.values())):
        print(f'"{nm}",' + ",".join(str(cnt[c]) for c in cols))


if __name__ == "__main__":
    main(*sys.argv[1:])
