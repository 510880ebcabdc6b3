"""Static SASS instruction count of a kernel by source function (dev tool): python tools/code_size.py <kernel substring> [binary]

binary: the library (default rrt_mpc_b200/libcudampc.so) or one translation unit's object, e.g. rrt_mpc_b200/_obj/tu7.o for the
register-form kernel (the library's kernel cubins share one name, so only the last one extracted from it is seen)."""
import re, subprocess, sys, os, tempfile, collections, bisect
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = os.path.abspath(sys.argv[2]) if len(sys.argv) > 2 else os.path.join(ROOT, "rrt_mpc_b200", "libcudampc.so"); kern = sys.argv[1]
tmp = tempfile.mkdtemp()
subprocess.run(["cuobjdump", "-xelf", "all", so], cwd=tmp, check=True, capture_output=True)
dis = []                       # every cubin of the library (one per translation unit)
for cub in sorted(f for f in os.listdir(tmp) if f.endswith(".cubin")):
    dis += subprocess.run(["nvdisasm", "-g", "-c", os.path.join(tmp, cub)], capture_output=True, text=True).stdout.splitlines()
csrc = os.path.join(ROOT, "rrt_mpc_b200", "csrc"); fmap = {}
for fn in os.listdir(csrc):
    st = []
    for i, ln in enumerate(open(os.path.join(csrc, fn)), 1):
        m = re.match(r"(?:template\s*<[^>]*>\s*)?(?:MPC_HD|__device__|__global__|static|inline)[^;(]*?([A-Za-z_0-9]+)\s*\(", ln)
        if m: st.append((i, m.group(1)))
    fmap[fn] = st
cnt = collections.Counter(); cur = None; infn = False; total = 0
for ln in dis:
    if ln.startswith(".text."): infn = kern in ln; continue
    if not infn: continue
    m = re.search(r'//## File "([^"]+)", line (\d+)', ln)
    if m: cur = (os.path.basename(m.group(1)), int(m.group(2))); continue
    if re.match(r'\s*/\*[0-9a-f]{4,}\*/\s+\S', ln):
        name = "?"
        if cur and cur[0] in fmap and fmap[cur[0]]:
            st = fmap[cur[0]]; j = bisect.bisect_right([a for a, _ in st], cur[1]) - 1
            name = f"{cur[0]}:{st[j][1]}" if j >= 0 else cur[0]
        elif cur: name = cur[0]
        cnt[name] += 1; total += 1
print(f"{kern}: {total} instructions = {total * 16 / 1024:.0f} KB")
for k, v in cnt.most_common(25): print(f"  {k:45s} {v:6d}  {v * 16 / 1024:6.1f} KB")
