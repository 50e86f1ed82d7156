#!/usr/bin/env python
"""SASS opcode histograms of the hot kernels of the built librisvec.so (cuobjdump, no GPU needed):
what proves which hardware paths a kernel uses (UTCHMMA = tcgen05.mma, STTM / LDTM = tcgen05.st / tcgen05.ld of
tensor memory, HMMA = mma.sync tensor path, UTMALDG / UTMASTG = TMA tensor loads / stores, SYNCS = mbarrier,
FFMA2 = packed fp32x2).  Writes profiles/r2_sass_histograms.md."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "ris_vec_marl_b200", "librisvec.so")
KERNELS = [("k_sarl_mma_tma<5>", r"k_sarl_mma_tmaILi5E"), ("k_sarl_mma<5,false>", r"k_sarl_mmaILi5ELb0E"),
           ("k_sarl_umma<8>", r"k_sarl_ummaILi8E"), ("k_sarl_mma_big<8>", r"k_sarl_mma_bigILi8E"), ("k_marl_tma", r"k_marl_tma"),
           ("k_sarl_v8<5,...,packed>", r"k_sarl_v8ILi5ELb1ELb1ELb1EE"), ("k_marl_v8<true,false>", r"k_marl_v8ILb1ELb0ELb0E"),
           ("k_sarl_cascade2<32,32,8>", r"k_sarl_cascade2ILi32ELi32ELi8E"), ("k_replay_store_flat<1>", r"k_replay_store_flatILi1E")]
MARK = ("HMMA", "UTMALDG", "UTMASTG", "SYNCS", "UBLKCP", "FFMA2", "FMUL2", "FADD2", "DADD", "DFMA", "DMUL", "MUFU", "SHFL", "LDS", "STS",
        "LDG", "STG", "BAR", "UTCHMMA", "UTCBAR", "LDTM", "STTM")


def main():
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    funcs, cur = {}, None
    for ln in sass.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1)
            funcs[cur] = collections.Counter()
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)", ln)
        if m and cur:
            funcs[cur][m.group(1)] += 1
    out = ["# SASS opcode histograms of the hot kernels (round 2)", "",
           "`python tools/sass_histogram.py` on the in-tree `librisvec.so` (nvcc 12.9, `-gencode arch=compute_100a,code=sm_100a`).",
           "Static instruction counts of the whole kernel (setup + every copy of the loop body).", ""]
    for label, pat in KERNELS:
        hit = [k for k in funcs if re.search(pat, k)]
        if not hit:
            out += [f"## {label}", "", "(not in this build)", ""]
            continue
        c = funcs[hit[0]]
        total = sum(c.values())
        out += [f"## {label}", "", f"`{hit[0][:110]}` -- {total} instructions", "",
                "| marker | count |", "|---|---|"]
        out += [f"| {k} | {c.get(k, 0)} |" for k in MARK if c.get(k, 0)]
        out += ["", "top opcodes: " + ", ".join(f"{k} {v}" for k, v in c.most_common(14)), ""]
    path = os.path.join(ROOT, "profiles", "r2_sass_histograms.md")
    with open(path, "w") as fh:
        fh.write("\n".join(out) + "\n")
    print(path)


if __name__ == "__main__":
    main()
