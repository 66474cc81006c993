#!/usr/bin/env python
"""SASS of the dense kernel instantiations of two builds of rtb_kernels.o, function by function (cuobjdump -sass):
identical, identical apart from constant-bank parameter offsets (c[0x0][...]), or different (with a short diff).  Kernels
that gained a LIST template parameter are matched to their dense (LIST = false) instantiation; list-mode and adaptive
kernels are skipped.

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

def norm_name(d, new):
    d = re.sub(r"^void ", "", d)
    d = d.split("(")[0]
    if new:
        d = re.sub(r"<false>$", "", d) if re.search(r"(generate_kernel|accumulate_kernel)<false>$", d) else d
        d = re.sub(r", false>$", ">", d) if re.search(r"(traverse_kernel|shade_kernel|tail_kernel)<", d) else d
    return d

def norm_ins(s):
    s = re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][P]", s)
    s = re.sub(r"0x[0-9a-f]+", "ADDR", s) if ("BRA" in s or "CALL" in s or "BSSY" in s) else s
    return s

old, new = funcs(sys.argv[1]), funcs(sys.argv[2])
oldn = {norm_name(dem(k), False): v for k, v in old.items()}
newn = {}
for k, v in new.items():
    d = dem(k)
    if (re.search(r"(traverse_kernel|shade_kernel|tail_kernel)<.*, true>", d) or re.search(r"(generate_kernel|accumulate_kernel)<true>", d) or "adaptive_" in d):
        continue
    newn[norm_name(d, True)] = v
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
for k in sorted(set(newn) - set(oldn)):
    print("NEW dense-named function:", k)
print(f"dense kernels: {len(oldn)}; identical {same}; identical apart from parameter offsets {diff_params}; different {diff}")
