#!/usr/bin/env python
"""Static SASS instruction counts per source line (and per opcode) of one kernel of liborbx.so.

  python tools/sass_lines.py k_describe_tma            # per-line histogram
  python tools/sass_lines.py k_describe_tma --ops      # opcode histogram

Needs the library built with -lineinfo (it is) and cuobjdump / nvdisasm on PATH.  CPU-only; used to budget
instruction counts before spending GPU time.
"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "rgbd_visualodometry_b200", "liborbx.so")


def main():
    pat = sys.argv[1]
    ops = "--ops" in sys.argv
    with tempfile.TemporaryDirectory() as td:
        subprocess.check_call(["cuobjdump", "-xelf", "all", SO], cwd=td, stdout=subprocess.DEVNULL)
        cubin = [f for f in os.listdir(td) if f.endswith(".cubin")][0]
        txt = subprocess.run(["nvdisasm", "--print-line-info", os.path.join(td, cubin)], capture_output=True, text=True).stdout
    cur_fn, cur_line = None, None
    per_line = collections.Counter()
    per_op = collections.Counter()
    total = collections.Counter()
    for ln in txt.splitlines():
        m = re.match(r"\s*\.section\s+\.text\.(\S+?),", ln)
        if m:
            cur_fn = m.group(1)
            cur_line = None
            continue
        if cur_fn is None or pat not in cur_fn:
            continue
        m = re.search(r'//## File "([^"]+)", line (\d+)', ln)
        if m:
            cur_line = (os.path.basename(m.group(1)), int(m.group(2)))
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", ln)
        if m:
            ins = m.group(1).strip()
            toks = ins.split()
            op = toks[1] if toks[0].startswith("@") and len(toks) > 1 else toks[0]
            op = op.split(".")[0]
            per_line[(cur_fn, cur_line)] += 1
            per_op[(cur_fn, op)] += 1
            total[cur_fn] += 1
    for fn, n in total.items():
        print(f"== {fn}: {n} instructions")
        if ops:
            for (f, op), c in sorted(per_op.items(), key=lambda kv: -kv[1]):
                if f == fn:
                    print(f"   {op:12s} {c}")
        else:
            for (f, l), c in sorted(per_line.items(), key=lambda kv: (kv[0][1] or ("", 0))):
                if f == fn:
                    print(f"   {l[0] if l else '?'}:{l[1] if l else 0:5d}  {c}")


if __name__ == "__main__":
    main()
