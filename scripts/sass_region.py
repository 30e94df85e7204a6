#!/usr/bin/env python
"""Lists the SASS of a source-line range of evaluate_kernel.cuh with executed counts and
stall samples: sass_region.py source.csv disasm.txt '<mangled kernel>' units first last"""
import csv, re, sys
src_csv, disasm, kernel, units, lo, hi = sys.argv[1], sys.argv[2], sys.argv[3], float(sys.argv[4]), int(sys.argv[5]), int(sys.argv[6])
instrs = []; inside = False; pending = []; cur = []
for line in open(disasm, errors='replace'):
    if line.startswith('\t.section\t.text.'):
        inside = line.startswith('\t.section\t.text.' + kernel + ','); continue
    if not inside: continue
    m = re.match(r'\s*//## File "([^"]+)", line (\d+)( inlined at)?', line)
    if m: pending.append((m.group(1).split('/')[-1], int(m.group(2)))); continue
    m = re.match(r'\s*/\*([0-9a-f]{4,})\*/\s+(.*?);', line)
    if m:
        if pending: cur = pending; pending = []
        instrs.append((m.group(2).strip(), cur))
rows = list(csv.reader(open(src_csv))); hdr = rows[1]; idx = {h: i for i, h in enumerate(hdr)}
body = [r for r in rows[2:] if len(r) >= len(hdr)]
# Every instruction of the kernel is inlined, ultimately, into a line of the kernel body, so its
# outermost frame lies there; helpers defined above the kernel (copies, checks, ForEachBlock)
# lie above the body.  The body starts at the first line of any outermost frame, and each
# instruction is attributed to its innermost frame inside the body: one line, so disjoint
# ranges split the instructions between them.
kernel_frames = lambda frames: [f for f in frames if f[0] == 'evaluate_kernel.cuh']
body_first = min(kernel_frames(fr)[-1][1] for _, fr in instrs if kernel_frames(fr))
for k, (r, (text, frames)) in enumerate(zip(body, instrs)):
    kb = [f for f in kernel_frames(frames) if f[1] >= body_first]
    if kb and lo <= kb[0][1] <= hi:
        print('%5d %5.2f %5s  %-28s %s' % (k, int(r[idx['Instructions Executed']]) / units, r[idx['# Samples']], '%s:%d' % frames[0], text[:72]))
