#!/usr/bin/env python
"""SASS of the kernel instantiations of two builds of rtb_kernels.o, function by function (cuobjdump -sass): identical,
identical apart from constant-bank parameter offsets (c[0x0][...]), or different (with a short diff).  Every kernel of the
old build is compared with the new build's instantiation of the same name, or, where the new build added template
parameters at the end (LIST, ENV), with the one whose added parameters are all false.  Instantiations only the new build
has are listed at the end.

    python tools/sass_diff.py OLD/build/rtb_kernels.o NEW/build/rtb_kernels.o
"""
import re, subprocess, sys

def funcs(obj):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    res, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if name: res[name] = body
            name, body = m.group(1), []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and name:
            body.append(m.group(1))
    if name: res[name] = body
    return res

def dem(n):
    return subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip()

def base_name(d):
    return re.sub(r"^void ", "", d).split("(")[0]

def strip_false(d):
    """The name with its last template argument removed when that argument is false (None otherwise)."""
    if d.endswith("<false>"):
        return d[: -len("<false>")]
    if d.endswith(", false>"):
        return d[: -len(", false>")] + ">"
    return None

def norm_ins(s):
    s = re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][P]", s)
    s = re.sub(r"0x[0-9a-f]+", "ADDR", s) if ("BRA" in s or "CALL" in s or "BSSY" in s) else s
    return s

old, new = funcs(sys.argv[1]), funcs(sys.argv[2])
oldn = {base_name(dem(k)): v for k, v in old.items()}
newn, extra = {}, []
for k, v in new.items():
    d = base_name(dem(k))
    m = d
    while m is not None and m not in oldn:
        m = strip_false(m)
    if m is None or m in newn:
        extra.append(d)
    else:
        newn[m] = v
same = diff_params = diff = 0
for k, v in sorted(oldn.items()):
    if k not in newn:
        print("MISSING in new:", k); diff += 1; continue
    w = newn[k]
    if v == w:
        same += 1
    elif [norm_ins(x) for x in v] == [norm_ins(x) for x in w]:
        diff_params += 1
    else:
        diff += 1
        import difflib
        d = list(difflib.unified_diff([norm_ins(x) for x in v], [norm_ins(x) for x in w], lineterm="", n=1))
        print("DIFF", k, len(v), len(w)); print("\n".join(d[:30]))
for k in sorted(extra):
    print("only in new:", k)
print(f"kernels of the old build: {len(oldn)}; identical {same}; identical apart from parameter offsets {diff_params}; different {diff}")
