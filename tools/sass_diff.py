"""Compare the binary32 kernels' SASS of two builds of libwrfb200.so, function by function.

    python tools/sass_diff.py OLD.so NEW.so      # exit 0 when every float kernel is identical

Instruction text and encodings are compared; code addresses and cuobjdump's column padding (which depends on the
longest instruction in the module) are stripped.  Used to show that a change leaves the float kernels untouched."""
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
        elif name and re.match(r"\s+/\*[0-9a-f]{4}\*/", ln):
            res[name].append(" ".join(re.sub(r"/\*[0-9a-f]{4,}\*/", "", ln).split()))
    return res


a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
sel = [n for n in a if re.search(r"amt_pipe_|amt_tile_kernel|amt_column_kernel", n) and "_r8" not in n]
bad = [n for n in sel if a[n] != b.get(n)]
print(f"{len(sel)} float kernels compared, {sum(len(a[n]) for n in sel)} instructions; differing: {bad}")
sys.exit(1 if bad else 0)
