#!/usr/bin/env python
"""SASS opcode evidence of the shipped library: per kernel, how many tcgen05 / TMEM / TMA / mbarrier / reduction
instructions `cuobjdump -sass scd_b200/libscd_b200.so` shows (the PTX names never appear in SASS:
tcgen05.mma -> UTC*MMA, tcgen05.ld/st -> LDTM/STTM, cp.async.bulk.tensor -> UTMALDG, tcgen05.commit -> UTCBAR,
mbarrier -> SYNCS).   python tools/sass_opcodes.py > profiles/r2_sass_opcodes.txt"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, 'scd_b200', 'libscd_b200.so')
PAT = re.compile(r'\b(UTC[A-Z0-9]*MMA(?:\.[A-Z0-9_]+)*|UTCBAR(?:\.[A-Z0-9_]+)*|LDTM(?:\.[A-Za-z0-9_]+)*|STTM(?:\.[A-Za-z0-9_]+)*|'
                 r'UTMALDG(?:\.[A-Z0-9_]+)*|UTCATOMSWS(?:\.[A-Z0-9_]+)*|SYNCS(?:\.[A-Z0-9_]+)*|REDG(?:\.[A-Z0-9_]+)*|'
                 r'HMMA(?:\.[A-Z0-9_]+)*|FMNMX3?|REDUX(?:\.[A-Z0-9_]+)*|ATOMS(?:\.[A-Z0-9_]+)*|ATOMG(?:\.[A-Z0-9_]+)*|UCGABAR_[A-Z]+|USETMAXREG(?:\.[A-Z0-9_]+)*)\b')


def main():
    sass = subprocess.run(['cuobjdump', '-sass', LIB], capture_output=True, text=True, check=True).stdout
    sha = subprocess.run(['sha1sum', LIB], capture_output=True, text=True).stdout.split()[0][:16]
    print(f'# cuobjdump -sass scd_b200/libscd_b200.so (sha1 {sha}), sm_100a: opcode counts per kernel')
    print('# UTC*MMA = tcgen05.mma (.2CTA = cta_group::2), LDTM / STTM = tcgen05.ld / st, UTMALDG = TMA tensor load,')
    print('# UTCBAR = tcgen05.commit, SYNCS = mbarrier, UTCATOMSWS = tcgen05.alloc, USETMAXREG = setmaxnreg, REDG = red.global, no HMMA (legacy mma.sync) anywhere')
    for f in re.split(r'\n\s*Function : ', sass)[1:]:
        name = f.split('\n', 1)[0].strip()
        dem = subprocess.run(['c++filt', name], capture_output=True, text=True).stdout.strip()
        n_instr = len(re.findall(r'/\*[0-9a-f]{4,}\*/\s+[A-Z@]', f))
        counts = collections.Counter(m.group(1) for m in PAT.finditer(f))
        print(f'\n## {dem.split("(")[0]}   ({n_instr} instructions)')
        for k, v in sorted(counts.items()):
            print(f'    {v:6d}  {k}')


if __name__ == '__main__':
    sys.exit(main())
