"""Innermost loops of a kernel in the shipped library, from `cuobjdump -sass`: every backward branch closes a loop; the
opcodes between its target and the branch are counted.  Used for the static side of DESIGN.md's roofline arguments (what
one trip of the decode GEMM's multiply loop issues, how many UBLKCP / UBLKPF the attention producer holds, ...).

    python scripts/sass_loops.py 'sgemm_dec_cluster_kernel<64, false, 8, 1, 3>' [more kernel-name substrings ...]
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "mt3_b200", "libmt3b200.so")


def kernels():
    sass = subprocess.run(["cuobjdump", "-sass", LIB], check=True, capture_output=True, text=True).stdout
    out, cur = collections.OrderedDict(), None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip() or m.group(1)
            cur = out.setdefault(re.sub(r"\(.*", "", name).replace("void ", ""), [])
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m and cur is not None:
            cur.append((int(m.group(1), 16), re.sub(r"^@!?U?P\w+\s+", "", m.group(2).strip())))
    return out


def loops(ins):
    for addr, txt in ins:
        if txt.startswith("BRA"):
            t = re.search(r"0x([0-9a-f]+)", txt)
            if t and int(t.group(1), 16) < addr:
                tgt = int(t.group(1), 16)
                body = [x for a, x in ins if tgt <= a <= addr]
                ops = collections.Counter(b.split()[0].split(".")[0] + (".128" if ".128" in b.split()[0] else "") for b in body)
                yield tgt, addr, len(body), ops


def main():
    pats = sys.argv[1:] or ["sgemm_dec_cluster_kernel<64, false, 8, 1, 3>"]
    ks = kernels()
    for name, ins in ks.items():
        if not any(p in name for p in pats):
            continue
        print(f"{name}: {len(ins)} instructions")
        for tgt, addr, n, ops in loops(ins):
            print(f"  loop 0x{tgt:04x}..0x{addr:04x}: {n:4d} instr  " + "  ".join(f"{k} {v}" for k, v in ops.most_common(8)))


if __name__ == "__main__":
    main()
