"""The "[psb]" lines of tools/r9a_calls.py's stderr with every number replaced by '#': the names and order of the
PSB_DEBUG_TIMING marks.  --sorted: sorted within each call (the two lanes of a large psb_align_pairs batch report
their passes in whichever order they finish)."""
import re
import sys

calls, cur = [], []
for line in open(sys.argv[1]):
    if not line.startswith("[psb]"):
        continue
    if line.startswith("[psb] == end of"):
        calls.append((line.strip(), cur))
        cur = []
        continue
    cur.append(re.sub(r"-?\d+(\.\d+)?", "#", line.rstrip()))
for end, lines in calls:
    for x in (sorted(lines) if "--sorted" in sys.argv else lines):
        print(x)
    print(end)
