"""SASS of every kernel of two builds of libgoldpolish_b200.so (cuobjdump -sass; addresses and encodings stripped):
instruction count and sha256 per function, parent first.  usage: python profiles/sass_compare.py PARENT.so THIS.so"""
import hashlib, re, subprocess, sys
def funcs(so):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    d, cur = {}, None
    for ln in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", ln)
        if m:
            cur = re.sub(r'_GLOBAL__N__[0-9a-f]+_\d+_(\w+?)_cu_[0-9a-f]+', r'(anon \1)', m.group(1)); d[cur] = []; continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", ln)
        if cur and m:
            d[cur].append(re.sub(r"\s+", " ", m.group(1)))
    return d
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
rows = []
for k in sorted(a):
    ha = hashlib.sha256("\n".join(a[k]).encode()).hexdigest()[:16]
    hb = hashlib.sha256("\n".join(b.get(k, [])).encode()).hexdigest()[:16] if k in b else "-"
    rows.append(f"  {'identical' if ha == hb else 'DIFFERENT'}  {len(a[k]):6d} / {len(b.get(k, [])):6d}  {ha}  {k}")
print("existing kernels: parent / this change SASS instructions, sha256[:16] of the parent's stream, name")
print("\n".join(rows))
print("added by this change:")
for k in sorted(set(b) - set(a)):
    print(f"  {len(b[k]):6d}  {k}")
