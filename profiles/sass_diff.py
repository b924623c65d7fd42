"""Compare the SASS of two builds of libcobel_b200.so function by function.

    python profiles/sass_diff.py OLD.so NEW.so [substring ...]

For each kernel (optionally only those whose demangled name contains one of the substrings) prints
``identical``, ``offsets +D`` when the instruction streams are the same except for kernel-parameter offsets
that moved by D bytes (``c[0x0][...]`` operands and the immediates of indexed parameter loads), or ``CHANGED``
with the instruction counts.  Needs cuobjdump and cu++filt of the CUDA toolkit; no GPU.
"""
import re
import subprocess
import sys

CUDA_BIN = '/usr/local/cuda/bin'
HEX = re.compile(r'0x[0-9a-f]+')


def functions(so):
    out = subprocess.run([CUDA_BIN + '/cuobjdump', '-sass', so], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r'\s+Function : (\S+)', line)
        if m:
            name = m.group(1)
            res[name] = []
        elif name and re.search(r'/\*[0-9a-f]{4,}\*/', line):
            res[name].append(re.sub(r'/\*[0-9a-f]{4,}\*/', '', line.split(';')[0]).strip())
    names = list(res)
    dem = subprocess.run([CUDA_BIN + '/cu++filt'], input='\n'.join(names), capture_output=True, text=True,
                         check=True).stdout.split('\n')
    return {d: res[m] for m, d in zip(names, dem)}


def compare(a, b):
    if a == b:
        return 'identical'
    if a is None or b is None:
        return 'only in %s' % ('new' if a is None else 'old')
    if len(a) != len(b):
        return 'CHANGED %d -> %d instructions' % (len(a), len(b))
    shifts = set()
    for x, y in zip(a, b):
        if x == y:
            continue
        if HEX.sub('#', x) != HEX.sub('#', y):
            return 'CHANGED (same count %d)' % len(a)
        shifts |= {int(v, 16) - int(u, 16) for u, v in zip(HEX.findall(x), HEX.findall(y)) if u != v}
    return 'offsets %s' % ','.join('%+d' % s for s in sorted(shifts)) if len(shifts) == 1 else 'CHANGED (immediates)'


def main():
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    keys = [k for k in sorted(set(old) | set(new)) if len(sys.argv) < 4 or any(s in k for s in sys.argv[3:])]
    for k in keys:
        print('%-9s %-9s %s  %s' % (len(old.get(k) or ()), len(new.get(k) or ()), compare(old.get(k), new.get(k)), k))


if __name__ == '__main__':
    main()
