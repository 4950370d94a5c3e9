#!/usr/bin/env python
"""
SASS evidence for the hot kernels: ``cuobjdump -sass`` of the in-tree library, one file per kernel under profiles/ plus a
mnemonic histogram (UTCIMMA = tcgen05.mma kind::i8, LDTM = tcgen05.ld, UBLKCP = cp.async.bulk, DMMA = mma.sync f64,
LDGSTS = cp.async).  No GPU needed.

    python tools/sass_extract.py [tag]
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "pygpso_b200", "libgpso_b200.so")
KERNELS = {
    "ozaki_screen_kernel_S2_all_pairs": "19ozaki_screen_kernelILi2ELi128ELb1EE",
    "ozaki_screen_kernel_S3_NT128": "19ozaki_screen_kernelILi3ELi128ELb0EE",
    "ozaki_kernel_S6_TRMM": "12ozaki_kernelILi6ELi0EE",
    "ozaki_kernel_S7_LAUUM": "12ozaki_kernelILi7ELi1EE",
    "ozaki_kernel_S8_GEMM": "12ozaki_kernelILi8ELi2EE",
    "crosscov_screen_kernel_M52_S2": "22crosscov_screen_kernelILi2ELi2ELi128EE",
    "crosscov_screen_kernel_M52_S3": "22crosscov_screen_kernelILi2ELi3ELi128EE",
    "crosscov_slices_kernel_M52_S6": "22crosscov_slices_kernelILi2ELi6EE",
    "factor_persistent_kernel": "24factor_persistent_kernel",
    "predict_trmm_kernel": "19predict_trmm_kernel",
}
KEY = ("UTCIMMA", "UTCHMMA", "UTCQMMA", "LDTM", "STTM", "UBLKCP", "UTMALDG", "DMMA", "LDGSTS", "SYNCS", "DFMA", "FFMA", "MUFU", "LDS", "STG", "LDG")


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else "r02"
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    blocks = re.split(r"(?=\t*Function : )", sass)
    summary = []
    for name, mangled in KERNELS.items():
        body = next((b for b in blocks if b.lstrip().startswith("Function : ") and mangled in b.split("\n", 1)[0]), None)
        if body is None:
            summary.append(f"{name}: NOT FOUND ({mangled})")
            continue
        ops = collections.Counter()
        for line in body.splitlines():
            m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
            if m:
                ops[m.group(1).split(".")[0]] += 1
        # keep the instruction lines only (cuobjdump prints a second line with the upper encoding word per instruction) and
        # stop at the end of the function
        keep = []
        for line in body.splitlines():
            if re.match(r"\s+/\* 0x[0-9a-f]{16} \*/\s*$", line):
                continue
            if line.startswith("Fatbin") or line.startswith("=") and keep:
                break
            keep.append(re.sub(r"\s+/\* 0x[0-9a-f]{16} \*/\s*$", "", line))
        with open(os.path.join(ROOT, "profiles", f"{tag}_sass_{name}.txt"), "w") as fh:
            fh.write("\n".join(keep) + "\n")
        total = sum(ops.values())
        keys = ", ".join(f"{k} {ops[k]}" for k in KEY if ops.get(k))
        summary.append(f"{name}: {total} instructions; {keys}")
    text = "\n".join(summary) + "\n"
    with open(os.path.join(ROOT, "profiles", f"{tag}_sass_summary.txt"), "w") as fh:
        fh.write("cuobjdump -sass pygpso_b200/libgpso_b200.so (sm_100a), per kernel: instruction count and the mnemonics that matter\n" + text)
    print(text)


if __name__ == "__main__":
    main()
