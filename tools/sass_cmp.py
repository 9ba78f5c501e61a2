#!/usr/bin/env python
"""Compare the SASS of kernels between two builds of a translation unit (DESIGN K16: K12 and the K13 step kernel must
compile to the same instructions when the pass is templated on the loss).

    python tools/sass_cmp.py OLD.cubin NEW.cubin NAME=NAME ... [--out profiles/k16_sass_cmp.txt]
    python tools/sass_cmp.py OLD.cubin NEW.cubin --all [--ptxas OLD.log NEW.log] [--out ...]

Each NAME=NAME pair names a kernel of the old and of the new cubin by a substring of its demangled name (the
anonymous-namespace hash of the file differs between builds and is dropped).  The instruction words are compared:
cuobjdump's `/*addr*/ MNEMONIC ... ; /* word */ /* word */` lines, including the encodings; nothing else.

--all compares every kernel of the two cubins, which must hold the same set of demangled names.  --ptxas also compares
the registers, stack frame and spills that `nvcc -Xptxas -v` printed for each kernel of the two builds."""
import argparse
import re
import subprocess
import sys

CUOBJDUMP = '/usr/local/cuda/bin/cuobjdump'


def kernels(cubin):
    text = subprocess.run([CUOBJDUMP, '-sass', cubin], check=True, capture_output=True, text=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            name = subprocess.run(['c++filt', m.group(1)], check=True, capture_output=True, text=True).stdout.strip()
            name = re.sub(r'\(anonymous namespace\)::', '', name)
            out[name] = []
            continue
        if name is not None and re.match(r'\s*(/\*[0-9a-f]{4,}\*/|/\* 0x)', line):
            out[name].append(line.strip())
    return out


def ptxas(log):
    """demangled kernel name -> the 'Function properties' and 'Used ... registers' lines of `nvcc -Xptxas -v`"""
    out, name = {}, None
    for line in open(log):
        m = re.search(r"(?:Function properties for|Compiling entry function ')(\w+)", line)
        if m:
            name = subprocess.run(['c++filt', m.group(1)], check=True, capture_output=True, text=True).stdout.strip()
            name = re.sub(r'\(anonymous namespace\)::', '', name)
            out.setdefault(name, [])
        elif name and re.search(r'stack frame|registers', line):
            out[name].append(re.sub(r'\s+', ' ', line.replace('ptxas info    :', '')).strip())
    return out


def pick(ks, sub):
    hits = [k for k in ks if sub in k]
    if len(hits) != 1:
        sys.exit('%r matches %d kernels: %s' % (sub, len(hits), hits))
    return hits[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('old')
    ap.add_argument('new')
    ap.add_argument('pairs', nargs='*')
    ap.add_argument('--all', action='store_true')
    ap.add_argument('--ptxas', nargs=2, metavar=('OLD_LOG', 'NEW_LOG'))
    ap.add_argument('--out')
    a = ap.parse_args()
    old, new = kernels(a.old), kernels(a.new)
    lines, same = [], True
    if a.all:
        if set(old) != set(new):
            same = False
            lines += ['only old: %s' % k for k in sorted(set(old) - set(new))]
            lines += ['only new: %s' % k for k in sorted(set(new) - set(old))]
        a.pairs += ['%s=%s' % (k, k) for k in sorted(set(old) & set(new))]
        lines.append('%d kernels in the old cubin, %d in the new' % (len(old), len(new)))
    res_o, res_n = (ptxas(a.ptxas[0]), ptxas(a.ptxas[1])) if a.ptxas else ({}, {})
    for pair in a.pairs:
        o, n = pair.split('=')
        ko, kn = (o, n) if a.all else (pick(old, o), pick(new, n))
        eq = old[ko] == new[kn]
        same &= eq
        if a.all:
            lines.append('%-12s %s (%d lines)' % ('identical' if eq else 'DIFFERENT', ko, len(old[ko])))
        else:
            lines.append('%-12s %s\n  old: %s (%d lines)\n  new: %s (%d lines)'
                         % ('identical' if eq else 'DIFFERENT', pair, ko, len(old[ko]), kn, len(new[kn])))
        if a.ptxas:
            ro, rn = res_o.get(ko), res_n.get(kn)
            req = ro is not None and ro == rn
            same &= req
            lines.append('  %s %s' % ('resources identical:' if req else 'RESOURCES DIFFER:', ' | '.join(ro or [])
                                      + ('' if req else ' vs ' + ' | '.join(rn or []))))
    text = '\n'.join(lines) + '\n'
    print(text, end='')
    if a.out:
        with open(a.out, 'a') as f:
            f.write(text)
    sys.exit(0 if same else 1)


if __name__ == '__main__':
    main()
