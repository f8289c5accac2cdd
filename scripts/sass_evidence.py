#!/usr/bin/env python
"""Per-kernel SASS instruction counts of the shipped library (runs on the CPU box):
    python scripts/sass_evidence.py > profiles/sass_evidence.md"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "transmf_ad_b200", "libtmf_sm100a.so")
COLS = [("UTC*MMA", r"UTC[A-Z]*MMA"), ("LDTM", r"LDTM"), ("UTMALDG", r"UTMALDG"), ("UBLKCP", r"UBLKCP"), ("UTCBAR", r"UTCBAR"),
        ("SYNCS", r"SYNCS"), ("HMMA", r"HMMA"), ("LDSM", r"LDSM"), ("LDGSTS", r"LDGSTS"), ("FFMA2/FADD2", r"F(FMA|ADD|MUL)2"),
        ("HMNMX2/HSET2", r"(HMNMX2|HSET2)"),
        ("float atomics", r"(ATOM|RED)[A-Z.]*\.(F32|F64|ADD\.F)"), ("int atomics (global)", r"(ATOMG|REDG|ATOM\.|RED\.)")]


def main():
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    names = subprocess.run(["c++filt"], input="\n".join(re.findall(r"Function : (\S+)", sass)), capture_output=True, text=True).stdout.split("\n")
    counts, order, cur, i = {}, [], None, 0
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = re.sub(r"\(.*", "", names[i]).strip()
            i += 1
            counts[cur] = collections.Counter()
            order.append(cur)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m and cur:
            op = m.group(1)
            for name, pat in COLS:
                if re.match(pat, op):
                    counts[cur][name] += 1
    print("# SASS evidence (round 2 final): `cuobjdump -sass transmf_ad_b200/libtmf_sm100a.so`, instruction counts per kernel\n")
    print("`UTC*MMA` = tcgen05.mma (`UTCHMMA`, kind::f16), `LDTM` = tcgen05.ld, `UTMALDG` = TMA tensor load (cp.async.bulk.tensor), `UBLKCP` = "
          "cp.async.bulk (conv1.0 image windows), `UTCBAR` = tcgen05.commit, `SYNCS` = mbarrier operations; `HMMA` = legacy mma.sync (the 16-row "
          "token-panel GEMMs of the fused transformer encoder and the tensor-core attention kernels: bf16 hi/lo split products -- DESIGN.md "
          "sections 10.4 / 10.10 for why not tcgen05 there), `LDSM` = ldmatrix, `LDGSTS` = cp.async, `FFMA2/FADD2` = packed fp32 pairs, "
          "`HMNMX2/HSET2` = packed bf16 max / compare (max-pool backward).\n")
    print("Floating-point atomics: only the CUDA-core bring-up kernels (`conv_direct.cu`).  Integer atomics: last-block tickets and the Adam "
          "step ticket.\n")
    print("| kernel | " + " | ".join(c[0] for c in COLS) + " |")
    print("|---|" + "---:|" * len(COLS))
    key = lambda k: (-counts[k]["UTC*MMA"], -counts[k]["HMMA"], k)
    for k in sorted(order, key=key):
        if not any(counts[k].values()):
            continue
        print(f"| `{k}` | " + " | ".join(str(counts[k][c[0]]) if counts[k][c[0]] else "" for c in COLS) + " |")


if __name__ == "__main__":
    main()
