"""Blackwell-native SASS mnemonics per kernel of libataxxzero.so (cuobjdump -sass) -> profiles/rNN_sass_evidence.txt

    python tools/sass_evidence.py > profiles/r02_sass_evidence.txt
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEEP = ("UTC", "UBLKCP", "LDTM", "STTM", "SYNCS", "UCGABAR", "REDUX", "REDG", "ATOMG", "ELECT", "FENCE", "DADD", "DFMA", "DMUL", "MUFU.RCP64H",
        "MUFU.RSQ64H", "LDG", "STG", "ACQBULK", "PREEXIT", "SHFL")
KERNELS = ("k_net_pair", "k_tree_tick", "k_walk", "k_samples", "k_convILi2", "k_wgradE")


def main():
    txt = subprocess.run(["cuobjdump", "-sass", os.path.join(ROOT, "ataxxzero_b200", "libataxxzero.so")], capture_output=True, text=True).stdout
    print("# SASS evidence (cuobjdump -sass ataxxzero_b200/libataxxzero.so, sm_100a): mnemonics per kernel")
    print("# UTCHMMA(.2CTA) = tcgen05.mma (cta_group::2), LDTM / STTM = tcgen05.ld / st, UBLKCP = cp.async.bulk (TMA), UTCBAR(.2CTA.MULTICAST) =")
    print("# tcgen05.commit, SYNCS = mbarrier, UCGABAR = cluster barrier, REDUX = warp reduction, REDG...F64.RN = fire-and-forget fp64")
    print("# reduction with round-to-nearest (tree backup), LDG...STRONG.GPU = ld.global.cg (node data is read through L2)")
    for f in re.split(r"\n\s*Function : ", txt)[1:]:
        name = f.split("\n", 1)[0]
        if not any(k in name for k in KERNELS):
            continue
        c = collections.Counter()
        for m in re.finditer(r"^\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", f, re.M):
            if m.group(1).startswith(KEEP):
                c[m.group(1)] += 1
        short = re.sub(r"_ZN\d+_GLOBAL__N__[0-9a-f_]+az_\w+?_cu_[0-9a-f]+", "", name)
        print("\n== %s" % short[:110])
        for op, n in sorted(c.items(), key=lambda kv: -kv[1])[:24]:
            print("  %6d %s" % (n, op))


if __name__ == "__main__":
    main()
