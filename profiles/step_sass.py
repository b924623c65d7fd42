"""Static instruction counts of the Dyna-Q step loop, read from the SASS of a build.

    python profiles/step_sass.py LIB.so [MANGLED_SUBSTRING ...]

For each matching kernel (default: the row-summary kernels ``dynaq_warp_kernel<A, PLAIN, false, SUM>``, A = 2, 3, 4)
finds the step loop -- the innermost backward branch whose body holds the stream refill (the Philox multiplier
0xCD9E8D57) -- and prints
  * ``null path``: the instructions a step issues from the loop head (the window check) to the back edge when it
    refills nothing, its online update changes nothing and its replay batch is all-null.  The walk takes every
    conditional forward branch that stays inside the loop (the refill skip, the refresh skip, the all-null exit of
    the replay) and falls through every other branch (divergence checks, loop exits);
  * ``refill``: the instructions of one refill, the region its branch skips;
  * ``loop``: the static size of the loop body outside the refill.
Needs cuobjdump of the CUDA toolkit; no GPU.
"""
import re
import subprocess
import sys

CUDA_BIN = '/usr/local/cuda/bin'
PHILOX_MUL = '-0x326172a9'          # 0xCD9E8D57 as the signed immediate of IMAD.WIDE.U32 / IMAD.HI.U32
DEFAULT = ['dynaq_warp_kernelILi2ELb1ELb0ELb1E', 'dynaq_warp_kernelILi3ELb1ELb0ELb1E',
           'dynaq_warp_kernelILi4ELb1ELb0ELb1E']


def kernels(path, subs):
    out = subprocess.run([CUDA_BIN + '/cuobjdump', '-sass', path], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r'\s+Function : (\S+)', line)
        if m:
            name = m.group(1) if any(s in m.group(1) for s in subs) else None
            if name:
                res[name] = []
            continue
        m = re.match(r'\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;', line)
        if name and m:
            res[name].append((int(m.group(1), 16), m.group(2)))
    return res


def branch(ins):
    """(predicated, target) of a direct branch, else None."""
    m = re.match(r'(@!?U?P\w+\s+)?BRA(\.U)?\s+(?:!?U?P\d\s*,\s*)?(0x[0-9a-f]+)$', ins)
    return (m.group(1) is not None, int(m.group(3), 16)) if m else None


def analyse(code):
    addr = [a for a, _ in code]
    at = {a: i for i, a in enumerate(addr)}
    loops = []
    for i, (a, ins) in enumerate(code):
        b = branch(ins)
        if b and b[1] <= a:
            lo, hi = at[b[1]], i
            if any(PHILOX_MUL in x for _, x in code[lo:hi]):
                loops.append((hi - lo, lo, hi))
    _, lo, hi = min(loops)
    refill = None
    for i in range(lo, hi):
        b = branch(code[i][1])
        if b and b[0] and code[i][0] < b[1] <= code[hi][0]:
            j = at[b[1]]
            if any(PHILOX_MUL in x for _, x in code[i + 1:j]):
                refill = (i + 1, j)
                break
    path, i = 0, lo
    while i <= hi:
        path += 1
        b = branch(code[i][1])
        if i == hi:
            break
        if b and not code[i][1].startswith('BRA.DIV') and code[i][0] < b[1] <= code[hi][0]:
            i = at[b[1]]
        else:
            i += 1
    n_refill = refill[1] - refill[0]
    return path, n_refill, (hi - lo + 1) - n_refill


def main():
    subs = sys.argv[2:] or DEFAULT
    for name, code in sorted(kernels(sys.argv[1], subs).items()):
        dem = subprocess.run([CUDA_BIN + '/cu++filt'], input=name, capture_output=True, text=True).stdout.strip()
        path, refill, loop = analyse(code)
        print('null path %4d   refill %4d   loop %5d   %s' % (path, refill, loop, dem))


if __name__ == '__main__':
    main()
