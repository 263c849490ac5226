"""Aggregate an ncu `--page source --csv` (SASS) export by CUDA source line using nvdisasm -g line info.
usage: sass_lines.py src.csv sim.sass mangled_kernel_name"""
import csv, re, sys, collections
src_csv, sass, kname = sys.argv[1:4]
# parse nvdisasm: list of (offset, line)
lines = open(sass).read().splitlines()
start = next(i for i, l in enumerate(lines) if l.startswith('.text.' + kname + ':'))
cur = None; off2line = {}
for l in lines[start + 1:]:
    if l.startswith('\t.section') or l.startswith('.text.'):
        break
    m = re.search(r'//## File "([^"]+)", line (\d+)', l)
    if m:
        cur = (m.group(1).split('/')[-1], int(m.group(2))); continue
    m = re.match(r'\s+/\*([0-9a-f]{4,})\*/\s+(.*);', l)
    if m:
        off2line[int(m.group(1), 16)] = (cur, m.group(2).strip())
rows = list(csv.reader(open(src_csv)))
hi = next(i for i, r in enumerate(rows) if 'Source' in r and 'Address' in r)
hdr = rows[hi]
ia, isrc, istall, iex = hdr.index('Address'), hdr.index('Source'), hdr.index('Warp Stall Sampling (All Samples)'), hdr.index('Instructions Executed')
base = None
agg = collections.defaultdict(lambda: [0, 0])
tot_ex = tot_st = 0
for r in rows[hi + 1:]:
    if len(r) <= iex: continue
    try:
        a = int(r[ia], 16); ex = int(r[iex] or 0); st = int(r[istall] or 0)
    except ValueError:
        continue
    if base is None: base = a
    loc = off2line.get(a - base, (None, ''))[0]
    agg[loc][0] += ex; agg[loc][1] += st; tot_ex += ex; tot_st += st
print('total warp-instructions', tot_ex, 'stall samples', tot_st)
# regions = the functions of swim_device.cuh, found by their definitions (a line at column 0 that opens one)
import os
srcp = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'swim_b200', 'csrc', 'swim_device.cuh')
src_lines = open(srcp).read().splitlines()
starts = []
for n, l in enumerate(src_lines, 1):
    if re.match(r'^(SWIM_HD|__device__|static __global__|__global__|template <)', l):
        txt = l if '(' in l and not l.startswith('template') else (l + ' ' + (src_lines[n] if n < len(src_lines) else ''))
        txt = re.sub(r'__launch_bounds__\([^)]*\)', '', txt)
        m = re.search(r'([A-Za-z_]\w*)\s*\(', re.sub(r'template <[^>]*>', '', txt))
        if m and m.group(1) not in ('defined',):
            if not starts or starts[-1][1] != m.group(1):
                starts.append((n, m.group(1)))
regions = [(name, a, (starts[k + 1][0] - 1 if k + 1 < len(starts) else len(src_lines))) for k, (a, name) in enumerate(starts)]
reg = collections.defaultdict(lambda: [0, 0])
for loc, (ex, st) in agg.items():
    name = 'other'
    if loc and loc[0] == 'swim_device.cuh':
        for n, a, b in regions:
            if a <= loc[1] <= b: name = n; break
    elif loc: name = loc[0]
    reg[name][0] += ex; reg[name][1] += st
for n, (ex, st) in sorted(reg.items(), key=lambda x: -x[1][0]):
    print(f'{n:16s} exec {ex:10d} {100*ex/tot_ex:5.1f}%   stalls {st:8d} {100*st/max(1,tot_st):5.1f}%')
print('--- top lines by executed')
for loc, (ex, st) in sorted(agg.items(), key=lambda x: -x[1][0])[:int(sys.argv[4]) if len(sys.argv) > 4 else 40]:
    print(f'{str(loc):32s} exec {ex:9d} {100*ex/tot_ex:5.1f}%  stalls {st:7d} {100*st/max(1,tot_st):5.1f}%')
if len(sys.argv) > 6:
    a, b = int(sys.argv[5]), int(sys.argv[6])
    print('--- lines', a, b)
    srcl = src_lines
    for loc, (ex, st) in sorted((x for x in agg.items() if x[0] and x[0][0] == 'swim_device.cuh' and a <= x[0][1] <= b), key=lambda x: x[0][1]):
        if ex > 150000 or st > 100:
            print(f'{loc[1]:5d} exec {ex/16/1000:7.1f}k/round stalls {st:6d} | {srcl[loc[1]-1].strip()[:110]}')
