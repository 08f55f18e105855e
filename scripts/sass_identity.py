"""Instruction-for-instruction comparison of two builds of libeqd_iegmn.so (`cuobjdump -sass`): every kernel of the first
library is matched by name (template arguments stripped) with the kernels of the second, and reported identical if one of
them has exactly the same instruction sequence (addresses stripped).  Used to show that adding a template parameter (e.g.
the DROPOUT instantiations) left the existing instantiations' machine code unchanged.

    python scripts/sass_identity.py OLD.so NEW.so
"""
import re
import subprocess
import sys
from collections import defaultdict


def functions(so):
    out = subprocess.run(['cuobjdump', '-sass', so], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur and re.match(r'\s*/\*[0-9a-f]{4}\*/', line):
            funcs[cur].append(re.sub(r'/\*[0-9a-f]{4}\*/', '', line).split(';')[0].strip())
    return funcs


def demangle(names):
    res = subprocess.run(['c++filt'], input='\n'.join(names), capture_output=True, text=True, check=True).stdout
    return dict(zip(names, res.splitlines()))


def base_name(demangled):
    n = demangled[5:] if demangled.startswith('void ') else demangled
    return re.sub(r'<.*', '', n.split('(')[0])


def main(old, new):
    a, b = functions(old), functions(new)
    da, db = demangle(list(a)), demangle(list(b))
    by_base = defaultdict(list)
    for n in b:
        by_base[base_name(db[n])].append(n)
    same = 0
    for n in sorted(a, key=lambda k: da[k]):
        hits = [c for c in by_base.get(base_name(da[n]), []) if b[c] == a[n]]
        tag = 'identical' if hits else 'DIFFERENT'
        same += bool(hits)
        print(f'{tag:9s} {len(a[n]):6d} instr  {da[n].split("(")[0]}' + (f'  == {db[hits[0]].split("(")[0]}' if hits else ''))
    print(f'{same} of {len(a)} kernels identical; {len(b) - len(a)} kernels only in {new}')
    return same == len(a)


if __name__ == '__main__':
    sys.exit(0 if main(sys.argv[1], sys.argv[2]) else 1)
