"""Warp-stall samples of an .ncu-rep source page aggregated by source function of fit_group.cuh (what
profiles/r2g_fit_group_g8_by_function.txt holds).  Usage (CPU box):
    ncu -i prof.ncu-rep --page source --csv > /tmp/src.csv
    cuobjdump -xelf all time_series_spark_b200/csrc/_build/fit_group_inst.o        # -> fit_group_inst.sm_100a.cubin
    nvdisasm -g -c fit_group_inst.sm_100a.cubin | awk '<keep the section of the captured kernel>' > /tmp/g8_lines.txt
    python tools/ncu_by_function.py
(the kernel must have been compiled with -lineinfo; paths are the ones used above)."""
import re, csv, sys, collections, os
# map offset -> (file, line, inline chain top function?) from nvdisasm -g output
cur=None; off2line={}
for ln in open('/tmp/g8_lines.txt'):
    m=re.search(r'//## File "([^"]+)", line (\d+)(.*)', ln)
    if m:
        cur=(m.group(1).split('/')[-1], int(m.group(2)), m.group(3)); continue
    m=re.match(r'\s+/\*([0-9a-f]{4,5})\*/\s+(.*?);', ln)
    if m:
        off2line[int(m.group(1),16)]=(cur, m.group(2))
rows=list(csv.reader(open('/tmp/src.csv')))
hdr=rows[1]; ia=hdr.index('Address'); isamp=hdr.index('# Samples'); iex=hdr.index('Instructions Executed')
cols={k:hdr.index(k) for k in ['stall_wait','stall_no_inst','stall_short_sb','stall_long_sb','stall_branch_resolving','stall_selected','stall_not_selected','stall_math','stall_dispatch']}
base=int(rows[2][ia],16)
# function ranges in fit_group.cuh by line numbers
src=open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'time_series_spark_b200', 'csrc', 'fit_group.cuh')).read().split('\n')
funcs=[]
for i,l in enumerate(src,1):
    m=re.match(r'(?:__device__|__global__|template).*?\b(g_\w+|gvdot|fit_group_kernel|day_features|gsum|gmax|gscan_excl\w*)\(', l)
    if m and ('__device__' in l or '__global__' in l): funcs.append((i,m.group(1)))
    elif re.match(r'__device__ __forceinline__ void (run)\(',l.strip()): funcs.append((i,'GPoint::run'))
    elif 'struct GPoint' in l: funcs.append((i,'GPoint'))
def fn_of(file,line):
    if file!='fit_group.cuh': return file
    name='?'
    for (i,n) in funcs:
        if i<=line: name=n
    return name
agg=collections.defaultdict(lambda: collections.Counter())
tot=collections.Counter()
for r in rows[2:]:
    off=int(r[ia],16)-base
    info=off2line.get(off)
    if info is None or info[0] is None: key='(unknown)'
    else:
        (f,l,extra),sass=info
        key=fn_of(f,l)
    s=int(r[isamp]); e=int(r[iex])
    agg[key]['samples']+=s; agg[key]['inst']+=e
    for k,c in cols.items(): agg[key][k]+=int(r[c])
    tot['samples']+=s; tot['inst']+=e
print(f"total samples {tot['samples']} inst {tot['inst']}")
for k,v in sorted(agg.items(), key=lambda kv:-kv[1]['samples']):
    print(f"{k:22s} samp {100*v['samples']/tot['samples']:5.1f}%  inst {100*v['inst']/tot['inst']:5.1f}%  cyc/inst {v['samples']/max(v['inst'],1)*tot['inst']/tot['samples']:.2f}x | " + ' '.join(f"{c[6:]}:{100*v[c]/max(v['samples'],1):.0f}" for c in cols))
