"""SASS opcode histogram of every cubin in libpermutect_b200.so (evidence for which kernels run on the tensor pipe):
    python profiles/sass_histogram.py > profiles/r2/sass_histogram.md
UTCHMMA = tcgen05.mma, HMMA = warp-level mma.sync, LDTM / STTM = tcgen05.ld / st, UBLKCP = cp.async.bulk, UTCBAR = tcgen05.commit, SYNCS = mbarrier,
FFMA2 / FADD2 / FMUL2 = paired FP32, LD = generic-address load."""
import collections, os, re, subprocess, sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = os.path.join(R, "permutect_b200", "csrc", "libpermutect_b200.so")
objdir = os.path.join(R, "permutect_b200", "csrc", "build")
KEY = ["UTCHMMA", "HMMA", "LDTM", "STTM", "UBLKCP", "UTCBAR", "SYNCS", "FFMA", "FFMA2", "FADD", "FADD2", "FMUL", "FMUL2", "MUFU", "LDL",
       "STL", "RED", "ATOMG", "SHFL", "LD", "LDS", "STS", "LDG", "STG"]
print("| object | kernel | " + " | ".join(KEY) + " | all |\n|---|---|" + "---|" * (len(KEY) + 1))
for obj in sorted(os.listdir(objdir)):
    if not obj.endswith(".o"):
        continue
    txt = subprocess.run(["cuobjdump", "-sass", os.path.join(objdir, obj)], capture_output=True, text=True).stdout
    cur, hist = None, collections.OrderedDict()
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip().split("(")[0][-60:]
            hist[cur] = collections.Counter()
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur:
            hist[cur][m.group(1).split(".")[0]] += 1
    for k, c in hist.items():
        if sum(c.values()) < 200:
            continue
        print(f"| {obj} | `{k}` | " + " | ".join(str(c.get(x, 0)) for x in KEY) + f" | {sum(c.values())} |")
