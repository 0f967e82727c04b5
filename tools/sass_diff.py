"""Compare the kernels' SASS of two builds of libwrfb200.so, function by function.

    python tools/sass_diff.py OLD.so NEW.so      # exit 0 when every kernel of each build has identical SASS in the other

Kernels are matched by their demangled name without the parameter list or an anonymous namespace: the hash nvcc
puts into the name of an anonymous namespace (`_GLOBAL__N__<hex>_`) depends on the path of the source file, and a
kernel whose parameters or linkage change is still the same kernel.  Instruction text and both 64-bit halves of
every encoding are compared; code addresses and cuobjdump's column padding (which depends on the longest
instruction in the module) are stripped.  A kernel found in only one build is paired with a kernel found in only the
other build whose SASS is identical and reported as renamed; the rest are listed separately."""
import re
import subprocess
import sys


def funcs(so):
    out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for ln in out.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            name = m.group(1)
            res[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,}\*/", ln):
            res[name].append(" ".join(re.sub(r"/\*[0-9a-f]{4,}\*/", "", ln).split()))
        elif name and res[name] and re.fullmatch(r"\s+/\* 0x[0-9a-f]{16} \*/", ln):
            res[name][-1] += " " + ln.strip()       # second half of the encoding: the scheduling control bits
    names = subprocess.run(["cu++filt"], input="\n".join(res), capture_output=True, text=True,
                           check=True).stdout.splitlines()
    return {re.sub(r"^void |<unnamed>::|\([^()]*\)$", "", d): res[m] for m, d in zip(res, names)}


a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
both = [n for n in a if n in b]
same = [n for n in both if a[n] == b[n]]
only_a = [n for n in a if n not in b]
only_b = [n for n in b if n not in a]
# a kernel found in one build only is paired with one found in the other build only whose SASS is identical
renamed = []
for n in only_a:
    m = next((m for m in only_b if a[n] == b[m]), None)
    if m is not None:
        renamed.append((n, m))
        only_b.remove(m)
only_a = [n for n in only_a if n not in dict(renamed)]
print(f"{len(both)} kernels in both builds, {len(same)} identical "
      f"({sum(len(a[n]) for n in same)} instructions); {len(renamed)} renamed, identical "
      f"({sum(len(a[n]) for n, _ in renamed)} instructions)")
for n, m in renamed:
    print(f"  renamed, identical: {n} -> {m}")
for title, names in (("differing", [n for n in both if a[n] != b[n]]), (f"only in {sys.argv[1]}", only_a),
                     (f"only in {sys.argv[2]}", only_b)):
    for n in names:
        print(f"  {title}: {n}" + (f" ({len(a[n])} -> {len(b[n])} instructions)" if n in a and n in b else ""))
sys.exit(0 if len(same) + len(renamed) == len(a) == len(b) else 1)
