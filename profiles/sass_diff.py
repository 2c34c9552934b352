"""SASS of the int8 pipeline's add / concat / avg-pool kernels in two builds of libpq_sm100.so, compared function by
function.

    python profiles/sass_diff.py PARENT.so NEW.so

Prints how many add_requant / concat_requant / avgpool_global functions of the first library compile to identical SASS
in the second (instruction text, addresses stripped), which functions only the second has, and how many other
functions differ."""
import re, subprocess, sys
def funcs(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    res, cur, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if cur: res[cur] = body
            cur, body = m.group(1), []
        elif cur and re.search(r"/\*[0-9a-f]{4}\*/", line):
            body.append(re.sub(r"/\*[0-9a-f]{4}\*/", "", line).split(";")[0].strip())
    if cur: res[cur] = body
    return res
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
old = [k for k in a if re.search(r"add_requant_kernel|concat_requant_(vec|scalar)_kernel|avgpool_global_kernel", k)]
same = [k for k in old if a[k] == b.get(k)]
print("parent add/concat/avgpool functions:", len(old), " identical SASS in new library:", len(same))
for k in old:
    if k not in same: print("DIFFERS:", k)
print("functions only in new library:", len(set(b) - set(a)))
for k in sorted(set(b) - set(a)): print("  new:", k)
print("other parent functions with differing SASS:", sum(1 for k in a if k not in old and a[k] != b.get(k)))
