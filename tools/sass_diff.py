#!/usr/bin/env python
"""SASS of the kernel instantiations of two builds, function by function (cuobjdump -sass): identical, identical apart from
constant-bank parameter offsets (c[0x0][...]), or different (with a short diff).  Each side is one or more objects (the
kernel objects of a build: rtb_kernels.o, rtb_shade.o, rtb_tail_*.o; an older build has rtb_kernels.o alone), split by
"--".  Every kernel of the old build is compared with the new build's kernel of the same name.  Names are compared with the
trailing bool arguments of a shade or tail kernel turned into its feature word (bit i = argument i, rtb_kernels.h), so a
build from before the word, and one from before a feature was added (its missing bools are 0), pairs with the word's
instantiations.  Kernels only the new build has are listed at the end.

    python tools/sass_diff.py OLD/build/rtb_kernels.o -- NEW/build/rtb_kernels.o NEW/build/rtb_shade.o NEW/build/rtb_tail_*.o
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

def feature_word(d):
    """rtb::shade_kernel<bools...> -> rtb::shade_kernel<word>, rtb::tail_kernel<MEDIA, STACK, bools...> ->
    rtb::tail_kernel<MEDIA, STACK, word>; every other name as it is.  (A word argument demangles as e.g. 5u.)"""
    m = re.fullmatch(r"(rtb::(?:shade_kernel|tail_kernel))<(.*)>", d)
    if not m:
        return d
    args = [a.strip() for a in m.group(2).split(",")]
    fixed = 2 if m.group(1) == "rtb::tail_kernel" else 0
    head, rest = args[:fixed], args[fixed:]
    if all(a in ("false", "true") for a in rest):
        word = sum(1 << i for i, a in enumerate(rest) if a == "true")
    else:
        (w,) = rest
        word = int(w.rstrip("uU"))
    return f"{m.group(1)}<{', '.join(head + [str(word)])}>"

def norm_ins(s):
    s = re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][P]", s)
    s = re.sub(r"0x[0-9a-f]+", "ADDR", s) if ("BRA" in s or "CALL" in s or "BSSY" in s) else s
    return s

def kernels(objs):
    res = {}
    for o in objs:
        for k, v in funcs(o).items():
            n = feature_word(base_name(dem(k)))
            if n in res:
                sys.exit(f"{n} is in more than one object of one side")
            res[n] = v
    return res

args = sys.argv[1:]
if "--" in args:
    i = args.index("--"); old_objs, new_objs = args[:i], args[i + 1:]
else:
    old_objs, new_objs = args[:1], args[1:]
oldn, newn = kernels(old_objs), kernels(new_objs)
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
extra = sorted(set(newn) - set(oldn))
for k in extra:
    print("only in new:", k)
print(f"kernels of the old build: {len(oldn)}; identical {same}; identical apart from parameter offsets {diff_params}; "
      f"different {diff}; only in new {len(extra)}")
