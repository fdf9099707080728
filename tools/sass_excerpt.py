#!/usr/bin/env python3
"""SASS evidence for the tensor-core kernels: for one instantiation each of score_dump_tc_kernel (score_tc.cu) and
gemm_bf16x3_2sm_kernel (gemm_tc.cu), every tcgen05 / TMA / TMEM / mbarrier instruction of the disassembly (cuobjdump
-sass of the in-tree objects) with its line number, plus mnemonic counts per kernel.

    python tools/sass_excerpt.py > profiles/rNN_sass_tcgen05.txt
"""
import re
import subprocess
from collections import Counter
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
BUILD = ROOT / "gat-recommendation_b200" / "build"
# the instantiations the bench runs: DIM = 256, k = 20, no exclusion lists; split-bf16 GEMM with 256-column tiles
WANT = {"score_tc.o": "score_dump_tc_kernelILi4ELi20ELb0E", "gemm_tc.o": "gemm_bf16x3_2sm_kernelILi2ELi256E"}
KEY = re.compile(r"\b(UTCHMMA|UTCQMMA|UTCBAR|UTCCP|UTMALDG|UTMASTG|UTMAREDG|UTMAPF|UTMACCTL|LDTM|STTM|SYNCS|UTCATOMSWS|"
                 r"FENCE|ELECT)\b")


def main():
    for obj, pattern in WANT.items():
        text = subprocess.run(["cuobjdump", "-sass", str(BUILD / obj)], capture_output=True, text=True).stdout
        blocks = re.split(r"\n\s*Function : ", text)
        for block in blocks[1:]:
            name = block.split("\n", 1)[0].strip()
            if pattern not in name:
                continue
            lines = block.split("\n")
            ops = Counter()
            shown = []
            for n, line in enumerate(lines):
                m = re.search(r"/\*[0-9a-f]{4}\*/\s+(.*?);", line)
                if not m:
                    continue
                inst = m.group(1).strip()
                mnemonic = inst.split()[1] if inst.startswith("@") else inst.split()[0]
                ops[mnemonic.split(".")[0]] += 1
                if KEY.search(inst):
                    shown.append(f"  {n:6d}  {inst}")
            print(f"=== {obj}: {name}")
            print(f"instructions: {sum(ops.values())}; tensor-core / TMA / TMEM / mbarrier mnemonics:")
            for k in sorted(ops):
                if KEY.search(k):
                    print(f"    {k:12s} x{ops[k]}")
            print("\n".join(shown))
            print()
            break


if __name__ == "__main__":
    main()
