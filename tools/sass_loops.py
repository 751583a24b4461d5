"""Static loop census of one kernel: every backward branch of its SASS with the instruction count of the loop body it closes.

usage: python tools/sass_loops.py <lib.so> <mangled-name-substring> [min_body]

Prints one line per loop (start, end, instructions, the most frequent mnemonics).  The strip walks of the fused kernels are the
loops with a few hundred instructions; the steady-state trip of a walk covers three row steps.
"""
import collections
import re
import subprocess
import sys


def kernel_sass(lib, pat):
    out = subprocess.run(["cuobjdump", "-sass", lib], check=True, capture_output=True, text=True).stdout
    rows, on = [], False
    for line in out.splitlines():
        if "Function :" in line:
            on = pat in line
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(.*?)\s*;?\s*(/\*.*)?$", line)
        if on and m:
            rows.append((int(m.group(1), 16), m.group(2).rstrip(" ;")))
    return rows


def main():
    lib, pat = sys.argv[1], sys.argv[2]
    min_body = int(sys.argv[3]) if len(sys.argv) > 3 else 40
    rows = kernel_sass(lib, pat)
    index = {a: i for i, (a, _) in enumerate(rows)}
    print(f"{pat}: {len(rows)} instructions")
    for i, (a, ins) in enumerate(rows):
        m = re.search(r"\bBRA(?:\.\S+)?\s+(?:!?U?P\w+,\s*)?0x([0-9a-f]+)", ins)
        if not m:
            continue
        t = int(m.group(1), 16)
        if t >= a or t not in index:
            continue
        body = rows[index[t]:i + 1]
        if len(body) < min_body:
            continue
        ops = collections.Counter(re.sub(r"^@!?U?P\w+\s+", "", x).split()[0] for _, x in body)
        top = ", ".join(f"{k} {v}" for k, v in ops.most_common(10))
        print(f"loop {t:05x}..{a:05x}: {len(body)} instructions | {top}")


if __name__ == "__main__":
    main()
