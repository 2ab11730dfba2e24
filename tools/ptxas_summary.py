"""Summarise registers / spills per kernel from the nvcc -Xptxas -v logs (development aid); by default the per-unit
logs the build leaves in feedback-gnn_b200/csrc/_build/."""
import glob, re, sys
paths = sys.argv[1:] or sorted(glob.glob("feedback-gnn_b200/csrc/_build/*.log"))
log = "".join(open(p).read() for p in paths)
cur = None
for line in log.splitlines():
    m = re.search(r"Compiling entry function '(\S+)'", line)
    if m:
        cur = m.group(1)
    m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
    if m:
        spill = m.groups()
    m = re.search(r"Used (\d+) registers", line)
    if m and cur:
        name = re.sub(r"^_ZN5fbgnn\d+", "", cur)
        print(f"{name[:60]:60s} regs={m.group(1):>4s} stack/spill={spill}")
        cur = None
