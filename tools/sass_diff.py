#!/usr/bin/env python3
"""Compare the SASS of selected kernels in two builds of liblcb200.so.

    python tools/sass_diff.py OLD.so NEW.so [--kernels k_sign k_verify k_vec_addsub k_pack k_unpack]

Kernels are matched by name and template arguments once the anonymous-namespace hashes are dropped.  A template
parameter added with a default is matched to the old instantiation when the new argument equals the default:
`k_sign<0>` to the old non-template `k_sign`, `k_verify<b, s, v, 0>` to the old `k_verify<b, s, v>` (pass
`--default-arg NAME=VALUE` for other kernels).  Instructions are compared after the address comments are removed.
Prints one line per kernel (NEW for instantiations the old build lacks) and exits 1 if a compared kernel differs or
an old kernel has no counterpart in the new build.
"""
import argparse
import re
import subprocess
import sys
from collections import OrderedDict

DEFAULTS = {'k_sign': '0', 'k_verify': '0'}


def demangle(names):
    out = subprocess.run(['cu++filt'], input='\n'.join(names), capture_output=True, text=True, check=True).stdout
    return out.splitlines()


def kernels(lib):
    """{mangled name: [normalised instruction lines]} of every function in the library."""
    sass = subprocess.run(['cuobjdump', '-sass', lib], capture_output=True, text=True, check=True).stdout
    funcs, cur = OrderedDict(), None
    for line in sass.splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        if cur is None:
            continue
        m = re.match(r'\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;?\s*(/\*.*\*/)?\s*$', line)
        if m and m.group(1):
            cur.append(m.group(1))
    return funcs


def key_of(demangled, wanted):
    """'k_verify<true, 11, 14>' for 'void lcb::(anonymous namespace)::k_verify<true, 11, 14>(...)', or None."""
    m = re.search(r'::(k_\w+)(<[^>]*>)?\(', demangled)
    if not m or m.group(1) not in wanted:
        return None
    args = [re.sub(r'^\((?:bool|int)\)', '', a.strip()) for a in m.group(2)[1:-1].split(',')] if m.group(2) else []
    return m.group(1), args


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('old')
    ap.add_argument('new')
    ap.add_argument('--kernels', nargs='+', default=['k_sign', 'k_verify', 'k_vec_addsub', 'k_pack', 'k_unpack'])
    ap.add_argument('--default-arg', action='append', default=[], help='NAME=VALUE: a trailing template argument '
                                                                          'added with this default')
    a = ap.parse_args()
    defaults = dict(DEFAULTS)
    defaults.update(dict(kv.split('=', 1) for kv in a.default_arg))
    wanted = set(a.kernels)

    def index(lib):
        funcs = kernels(lib)
        names = list(funcs)
        out = {}
        for mangled, dem in zip(names, demangle(names)):
            k = key_of(dem, wanted)
            if k:
                out[(k[0], tuple(k[1]))] = funcs[mangled]
        return out

    old, new = index(a.old), index(a.new)
    bad = 0
    matched = set()
    for (name, args), body in sorted(new.items()):
        cand = [(name, args)]
        if args and args[-1] == defaults.get(name):
            cand.append((name, args[:-1]))
        match = next((c for c in cand if c in old), None)
        label = f'{name}<{", ".join(args)}>' if args else name
        if match is None:
            print(f'NEW      {label} ({len(body)} instructions; no counterpart in the old build)')
            continue
        matched.add(match)
        same = old[match] == body
        bad += not same
        shown = f'{match[0]}<{", ".join(match[1])}>' if match[1] else match[0]
        print(f'{"SAME" if same else "DIFFERS":8} {label} vs {shown} ({len(body)} / {len(old[match])} instructions)')
    for name, args in sorted(set(old) - matched):
        bad += 1
        print(f'MISSING  {name}<{", ".join(args)}> (only in the old build)' if args else f'MISSING  {name}')
    sys.exit(1 if bad else 0)


if __name__ == '__main__':
    main()
