"""Static SASS instruction count per source line / function of one kernel (needs -lineinfo).
usage: python tools/sass_by_line.py <lib.so> <mangled kernel name> [top]"""
import collections, os, re, subprocess, sys, tempfile
lib, kern = sys.argv[1], sys.argv[2]
top = int(sys.argv[3]) if len(sys.argv) > 3 else 40
tmp = tempfile.mkdtemp()
subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=tmp, capture_output=True)
cub = [f for f in os.listdir(tmp) if "kernels" in f][0]
txt = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(tmp, cub)], capture_output=True, text=True).stdout.split("\n")
start = [i for i, l in enumerate(txt) if l.startswith(f".text.{kern}:")][0]
end = next(i for i, l in enumerate(txt) if i > start and l.startswith("//--------------------- "))
cur = None
cnt = collections.Counter()
for l in txt[start:end]:
    m = re.match(r'\s*//## File "([^"]+)", line (\d+)', l)
    if m:
        cur = (os.path.basename(m.group(1)), int(m.group(2)))
    elif re.match(r"\s+/\*[0-9a-f]+\*/", l):
        cnt[cur] += 1
total = sum(cnt.values())
print("total", total)
# function map from source files
fmap = {}
for f in set(k[0] for k in cnt if k):
    path = None
    for root in ("aerobulk_b200/csrc",):
        p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), root, f)
        if os.path.exists(p):
            path = p
    if not path:
        continue
    name = "?"
    for n, line in enumerate(open(path), 1):
        m = re.match(r"^(?:template.*\n)?(?:ABD|ABM_FN|__global__|__device__|static)[^(;]*?(\w+)\s*\(", line)
        if m and not line.startswith(" "):
            name = m.group(1)
        fmap[(f, n)] = name
byfn = collections.Counter()
for k, v in cnt.items():
    byfn[(k[0], fmap.get(k, "?")) if k else ("?", "?")] += v
for k, v in byfn.most_common(top):
    print(f"{v:6d} {100*v/total:5.1f}%  {k[0]}:{k[1]}")
