#!/usr/bin/env python
"""Compare the device code of two builds of the library, kernel by kernel.
    python tools/sass_compare.py before/libgtscaffold_b200.so after/libgtscaffold_b200.so
Instructions are compared as cuobjdump -sass prints them, without addresses and encodings; a kernel
only one build has whose code equals a kernel only the other has is reported as renamed."""
import collections
import os
import re
import subprocess
import sys

BIN = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")


def name(line):
    """'void ns::k<(int)8>(ns::Args, unsigned int)' -> 'ns::k<(int)8>': drop the return type and the parameter list"""
    s, depth = line.removeprefix("void "), 0
    for i in range(len(s) - 1, -1, -1):
        depth += {")": 1, "(": -1}.get(s[i], 0)
        if depth == 0:
            return s[:i] if s.endswith(")") else s
    return s


def kernels(lib):
    sass = subprocess.run([os.path.join(BIN, "cuobjdump"), "-sass", lib], capture_output=True, text=True,
                          check=True).stdout
    sass = subprocess.run([os.path.join(BIN, "cu++filt")], input=sass, capture_output=True, text=True,
                          check=True).stdout
    code, body = collections.defaultdict(list), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (.*)$", line)
        if m:
            body = []
            code[name(m.group(1))].append(body)     # a kernel of a shared header is in every unit that launches it
        elif body is not None:
            m = re.match(r"\s*/\*[0-9a-f]+\*/\s*(.*?)\s*;", line)     # "/*0120*/  INSTR ... ;  /* 0x... */"
            if m:
                body.append(m.group(1))
    return {k: sorted("\n".join(b) for b in v) for k, v in code.items()}


a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
gone, new = sorted(set(a) - set(b)), sorted(set(b) - set(a))
renamed = [(x, y) for x in gone for y in new if a[x] == b[y]]
print("only before:", ", ".join(x for x in gone if x not in {p[0] for p in renamed}) or "none")
print("only after:", ", ".join(y for y in new if y not in {p[1] for p in renamed}) or "none")
print("renamed, same code:", ", ".join(f"{x} -> {y}" for x, y in renamed) or "none")
print("changed:", ", ".join(k for k in sorted(set(a) & set(b)) if a[k] != b[k]) or "none")
print(f"kernels: {sum(map(len, a.values()))} before, {sum(map(len, b.values()))} after")
