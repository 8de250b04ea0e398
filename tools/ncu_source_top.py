"""Per-source-line stall-sample totals of one kernel of an Nsight Compute report (compiled with -lineinfo, captured
with --import-source on), read on the CPU box:
  python tools/ncu_source_top.py prof_attn.ncu-rep attn_bwd_row2_kernel [N]"""
import csv
import io
import re
import subprocess
import sys
from collections import defaultdict


def main():
    path, kernel = sys.argv[1], sys.argv[2]
    top = int(sys.argv[3]) if len(sys.argv) > 3 else 25
    out = subprocess.run(["ncu", "-i", path, "--page", "source", "--csv", "--kernel-name", f"regex:{kernel}", "--print-source", "sass"],
                         capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(out)))
    hdr = None
    for i, r in enumerate(rows):
        if "Source" in r and any("Sampl" in c for c in r):
            hdr, body = r, rows[i + 1:]
            break
    if hdr is None:
        print(out[:2000])
        return
    col = {}
    for i, c in enumerate(hdr):
        col.setdefault(c, i)
    samp = "Warp Stall Sampling (All Samples)"
    exe = "Instructions Executed"
    stall_cols = [c for c in hdr if c.startswith("stall_") and "Not Issued" not in c]
    stall_tot = defaultdict(int)
    tot = 0
    ops = defaultdict(lambda: [0, 0])
    lines = []
    for r in body:
        if len(r) <= col[samp]:
            continue
        try:
            s = int(r[col[samp]].replace(",", "") or 0)
        except ValueError:
            continue
        e = 0
        if exe is not None:
            try:
                e = int(r[col[exe]].replace(",", "") or 0)
            except (ValueError, IndexError):
                pass
        src = r[col["Source"]]
        m = re.match(r"\s*(@!?U?P\d+\s+)?([A-Z0-9_.]+)", src)
        op = m.group(2).split(".")[0] if m else "?"
        ops[op][0] += s
        ops[op][1] += e
        tot += s
        why = []
        for c in stall_cols:
            try:
                v = int(r[col[c]].replace(",", "") or 0)
            except (ValueError, IndexError):
                v = 0
            stall_tot[c] += v
            if v:
                why.append((v, c[6:]))
        why.sort(reverse=True)
        lines.append((s, e, src.strip()[:84] + "   [" + ", ".join(f"{n} {v}" for v, n in why[:2]) + "]"))
    print(f"kernel {kernel}: {tot} stall samples, {sum(v[1] for v in ops.values())} warp-level instructions executed")
    print("stall reasons: " + ", ".join(f"{c[6:]} {v}" for c, v in sorted(stall_tot.items(), key=lambda kv: -kv[1])[:9]))
    print("\nby opcode (samples, executed):")
    for op, (s, e) in sorted(ops.items(), key=lambda kv: -kv[1][0])[:18]:
        print(f"  {op:14s} {s:8d} {100.0 * s / max(tot, 1):5.1f}%   exec {e}")
    print(f"\ntop {top} instructions by samples:")
    for s, e, src in sorted(lines, reverse=True)[:top]:
        print(f"  {s:7d} {100.0 * s / max(tot, 1):5.1f}%  exec {e:9d}  {src}")


if __name__ == "__main__":
    main()
