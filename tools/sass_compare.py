"""Compare the SASS of every kernel in an object file built at a parent commit with its counterpart in a new build.

    python tools/sass_compare.py PARENT.o NEW.o

Instructions are compared with addresses, encodings and line information stripped.  Kernels that gained a feature-type
template parameter are matched to their float32 instantiation (fp_front_kernel<G> -> <G, 0>,
inv_{gather,long}_kernel<V> -> <0, V>)."""
import re, subprocess, sys
def funcs(obj):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    fs, cur, name = {}, [], None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name: fs[name] = cur
            name, cur = m.group(1), []
            continue
        if name is None: continue
        t = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)          # addresses
        t = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", t)             # encodings
        t = t.strip()
        if t and not t.startswith("//") and not t.startswith(".") : cur.append(t)
    if name: fs[name] = cur
    return fs
def key(d):
    return d[:d.index(">(") + 1] if ">(" in d else d.split("(")[0]
def dem(names):
    r = subprocess.run(["/usr/local/cuda/bin/cu++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, r))
old, new = funcs(sys.argv[1]), funcs(sys.argv[2])
do, dn = dem(list(old)), dem(list(new))
rev = {key(v): k for k, v in dn.items()}
def mapname(d):
    d = re.sub(r"fp_front_kernel<\(int\)(\d+)>", r"fp_front_kernel<(int)\1, (int)0>", d)
    d = re.sub(r"inv_(gather|long)_kernel<\(bool\)(\d)>", r"inv_\1_kernel<(int)0, (bool)\2>", d)
    return d
same = diff = 0
for k, body in old.items():
    nd = key(mapname(do[k]))
    if nd not in rev:
        print("MISSING", do[k]); diff += 1; continue
    if new[rev[nd]] == body: same += 1
    else:
        diff += 1; print("DIFFERS", do[k], len(body), len(new[rev[nd]]))
print(f"{sys.argv[1]}: {same} float32 kernels identical, {diff} differ/missing; new build has {len(new)} functions, parent {len(old)}")
