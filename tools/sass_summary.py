#!/usr/bin/env python3
"""Static SASS statistics of the hot kernels (cuobjdump -sass on the objects built in-tree): instruction mix per kernel and
an excerpt of one Montgomery product, so that claims like "every 32x32 limb product is one IMAD.WIDE.U32(.X)" can be checked
from the tree.      python tools/sass_summary.py > profiles/r2_sass_summary.txt"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "simpleworks_b200", "_build")
KERNELS = {"msm_pairs.o": ["k_pair_bwd", "k_pair_fwd", "k_pair_inv"], "msm_accumulate.o": ["k_msm_accumulate"], "ntt.o": ["k_ntt_pass"], "msm_sort.o": ["k_msm_digitsILb1ELi23E", "k_msm_digitsILb0ELi20E"],
           "vec.o": ["k_mul_peak", "k_fq_mul", "k_fr_mul"]}


def functions(obj):
    out = subprocess.run(["cuobjdump", "-sass", os.path.join(BUILD, obj)], capture_output=True, text=True).stdout
    cur, body = None, {}
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            body[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            body[cur].append(line)
    return body


def opcode(line):
    m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    return m.group(1) if m else None


def main():
    for obj, names in KERNELS.items():
        if not os.path.exists(os.path.join(BUILD, obj)):
            continue
        for fn, lines in functions(obj).items():
            if not any(n in fn for n in names):
                continue
            mix = collections.Counter(opcode(l) for l in lines)
            mix.pop(None, None)
            total = sum(mix.values())
            wide = sum(v for k, v in mix.items() if k.startswith("IMAD.WIDE"))
            split = sum(v for k, v in mix.items() if k in ("IMAD", "IMAD.HI.U32", "IMAD.U32") or k.startswith("IMAD.HI"))
            print(f"== {obj}: {fn}")
            print(f"   {total} SASS instructions; IMAD.WIDE* {wide} ({100.0 * wide / total:.1f} %), other IMAD* {split}, "
                  f"LDG {sum(v for k, v in mix.items() if k.startswith('LDG'))}, STG {sum(v for k, v in mix.items() if k.startswith('STG'))}, "
                  f"LDS {sum(v for k, v in mix.items() if k.startswith('LDS'))}, BAR {sum(v for k, v in mix.items() if k.startswith('BAR'))}, "
                  f"SHFL {sum(v for k, v in mix.items() if k.startswith('SHFL'))}, local LDL/STL {sum(v for k, v in mix.items() if k in ('LDL', 'STL') or k.startswith('LDL.') or k.startswith('STL.'))}")
            print("   top opcodes: " + ", ".join(f"{k} {v}" for k, v in mix.most_common(8)))
            if "k_pair_bwd" in fn and "Lb1" in fn:
                # one Fq Montgomery product: the first run of ~300 consecutive instructions dominated by IMAD.WIDE
                start = next((i for i, l in enumerate(lines) if "IMAD.WIDE" in l), 0)
                print("   excerpt (start of the first Fq Montgomery product, 40 instructions):")
                for l in lines[start:start + 40]:
                    print("      " + re.sub(r"\s+/\* 0x[0-9a-f]+ \*/\s*$", "", l.rstrip())[:110])
            print()


if __name__ == "__main__":
    main()
