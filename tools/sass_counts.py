"""Per-function SASS counts of a CUDA object file: instructions, DMMA, LDL / STL (local-memory spills), SHFL and BAR.

    python tools/sass_counts.py bilevel-gait-gen_b200/build/bgg_ipm.o

One line per function, in the order cuobjdump lists them; then, for each kernel, the body plus every function it reaches
through calls (the call graph comes from the call relocations of the object's .rela.text sections).  This is the code a
warp may have to fetch while it runs the kernel.  Names lose the file-internal namespace prefix that nvcc puts on static
functions.  Needs cuobjdump (CUDA_HOME or /usr/local/cuda), no GPU.
"""
import os
import re
import subprocess
import sys
from collections import OrderedDict

KINDS = ("DMMA", "LDL", "STL", "SHFL", "BAR")
CALL_RELOC = "R_CUDA_ABS55_16_34"   # the relocation of a CALL.ABS target


def cuobjdump(obj, flag):
    exe = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    return subprocess.run([exe, flag, obj], check=True, capture_output=True, text=True).stdout


def count_sass(text):
    funcs = OrderedDict()
    cur = None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = funcs.setdefault(m.group(1), dict(insts=0, **{k: 0 for k in KINDS}))
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[0-9T]\s+)?([A-Z0-9_]+)", line)
        if cur is None or not m:
            continue
        cur["insts"] += 1
        op = m.group(1)
        for k in KINDS:
            if op == k:
                cur[k] += 1
    return funcs


def call_graph(elf_text, names):
    calls = {n: set() for n in names}
    cur = None
    for line in elf_text.splitlines():
        m = re.match(r"\.section \.rela\.text\.(\S+)", line)
        if m:
            cur = m.group(1) if m.group(1) in calls else None
            continue
        if line.startswith(".section"):
            cur = None
            continue
        f = line.split()
        if cur is not None and len(f) >= 3 and f[2] == CALL_RELOC and f[1] in calls and f[1] != cur:
            calls[cur].add(f[1])
    return calls


def reach(calls, root):
    seen, todo = set(), [root]
    while todo:
        for c in calls[todo.pop()]:
            if c not in seen:
                seen.add(c)
                todo.append(c)
    return seen


def short(name):
    return re.sub(r"^_ZN\d+_INTERNAL_\w+?_\d+_\w+?_cu_[0-9a-f]+3bgg", "", name)


def main(obj):
    funcs = count_sass(cuobjdump(obj, "-sass"))
    calls = call_graph(cuobjdump(obj, "-elf"), funcs)
    for name, c in funcs.items():
        print(short(name), f"insts={c['insts']}", " ".join(f"{k}={c[k]}" for k in KINDS))
    called = set().union(*calls.values()) if calls else set()
    for name in funcs:
        if name in called:
            continue
        callees = reach(calls, name)
        tot = {k: funcs[name][k] + sum(funcs[c][k] for c in callees) for k in ("insts",) + KINDS}
        print(f"total {short(name)} (body + {len(callees)} callees) insts={tot['insts']}", " ".join(f"{k}={tot[k]}" for k in KINDS))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
