#!/usr/bin/env python
"""Static opcode histogram of the per-pixel loop of one kernel (no GPU needed):

    python tools/sass_hist.py [--by-callsite] [object-or-cubin] [kernel-name-substring]

Defaults: planetmapper_b200/csrc/build/backplane_kernels.o and the single-frame image kernel of
the default surface stack on a spin-symmetric body (backplanes_img_param_kernel<false, kDefaultStackMask, true>).  The loop body
is the span from the target of the kernel's widest backward branch to that branch.  Besides the
opcode counts it prints the numbers the FP64 issue model cares about: DFMAs whose three sources
are all ordinary registers (they hold the issue port for 3 cycles instead of 2), the FSEL pairs of
double selects, and the constant / uniform moves (LDC, LDCU, UMOV) that feed them.

--by-callsite attributes the loop's instructions to the statements of image_pixel they were inlined
from (nvdisasm -g -gi line info of the object's cubin), weighted by the issue rules of DESIGN.md
section 3.4: 3 cycles for a DFMA with three register sources, 2 for any other FP64 instruction, 1 for
everything else (the upper end of the measured 0.5 - 1).  Out-of-line callees count as their CALL.
"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_OBJ = os.path.join(ROOT, 'planetmapper_b200', 'csrc', 'build', 'backplane_kernels.o')
DEFAULT_KERNEL = 'backplanes_img_param_kernelILb0ELm1044495ELb1E'
FP64 = ('DFMA', 'DMUL', 'DADD', 'DSETP', 'DMNMX')

INSN = re.compile(r'/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)\s*([^;]*);')
REG = re.compile(r'^-?\|?R\d+\|?(\.reuse)?$')


def kernel_sass(obj, kernel):
    sass = subprocess.run(['cuobjdump', '-sass', obj], capture_output=True, text=True, check=True).stdout
    funcs = re.split(r'\n\s*Function : ', sass)
    hits = [f for f in funcs[1:] if kernel in f.split('\n', 1)[0]]
    if len(hits) != 1:
        sys.exit('%d functions match %r' % (len(hits), kernel))
    insns = []
    for m in INSN.finditer(hits[0]):
        insns.append((int(m.group(1), 16), m.group(3), m.group(4).strip()))
    return hits[0].split('\n', 1)[0].strip(), insns


def loop_body(insns):
    """instructions between the target of the widest backward branch and the branch itself"""
    best = None
    for addr, op, args in insns:
        if op.startswith('BRA'):
            m = re.search(r'0x([0-9a-f]+)\s*$', args)
            if m and int(m.group(1), 16) < addr:
                span = (int(m.group(1), 16), addr)
                if best is None or span[1] - span[0] > best[1] - best[0]:
                    best = span
    if best is None:
        sys.exit('no backward branch')
    return best, [i for i in insns if best[0] <= i[0] <= best[1]]


def issue_cycles(op, args):
    base = op.split('.')[0]
    if base == 'DFMA' and all(REG.match(a.strip()) for a in args.split(',')[1:]):
        return 3
    return 2 if base in FP64 else 1


CALLER = re.compile(r'//## File "[^"]*pm_device\.cuh", line (\d+) inlined at "[^"]*backplane_kernels\.cu"')


def callsite_table(obj, name, lo, hi):
    """{pm_device.cuh line of image_pixel: Counter(insns, fp64, dfma3r, cycles)} over the loop lo..hi"""
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run(['cuobjdump', '-xelf', 'all', os.path.abspath(obj)], cwd=tmp, check=True, capture_output=True)
        cubins = [f for f in os.listdir(tmp) if f.endswith('.cubin')]
        if len(cubins) != 1:
            sys.exit('expected one cubin in %s, found %s' % (obj, cubins))
        text = subprocess.run(['nvdisasm', '-g', '-gi', os.path.join(tmp, cubins[0])], capture_output=True,
                              text=True, check=True).stdout
    start = text.find('\n.text.%s:' % name)
    if start < 0:
        sys.exit('function %s not found by nvdisasm' % name)
    end = text.find('\t.section', start)
    table = collections.defaultdict(collections.Counter)
    chain, fresh = [], True
    for line in text[start:end if end > 0 else len(text)].split('\n'):
        if line.lstrip().startswith('//## File'):
            if fresh:
                chain, fresh = [], False
            chain.append(line)
            continue
        m = INSN.search(line)
        if not m:
            continue
        fresh = True
        addr = int(m.group(1), 16)
        if not lo <= addr <= hi:
            continue
        site = next((int(c.group(1)) for c in map(CALLER.search, chain) if c), 0)
        op, args = m.group(3), m.group(4)
        row = table[site]
        row['insns'] += 1
        row['fp64'] += op.split('.')[0] in FP64
        row['dfma3r'] += issue_cycles(op, args) == 3
        row['cycles'] += issue_cycles(op, args)
    return table


def print_callsites(obj, name, lo, hi):
    table = callsite_table(obj, name, lo, hi)
    src = open(os.path.join(ROOT, 'planetmapper_b200', 'csrc', 'pm_device.cuh')).read().split('\n')
    total = sum(r['cycles'] for r in table.values())
    print('issue-weighted cycles of the loop: %d (DFMA 3R = 3, other FP64 = 2, rest = 1)' % total)
    print('%6s %6s %5s %6s %6s  %s' % ('cycles', 'share', 'insns', 'fp64', 'dfma3r', 'image_pixel call site (pm_device.cuh)'))
    for site, r in sorted(table.items(), key=lambda kv: -kv[1]['cycles']):
        where = '%d: %s' % (site, src[site - 1].strip()[:70]) if site else '(kernel / img_tile, outside image_pixel)'
        print('%6d %5.1f%% %5d %6d %6d  %s' % (r['cycles'], 100.0 * r['cycles'] / total, r['insns'], r['fp64'],
                                                r['dfma3r'], where))


def main():
    args = sys.argv[1:]
    by_callsite = '--by-callsite' in args
    args = [a for a in args if a != '--by-callsite']
    obj = args[0] if len(args) > 0 else DEFAULT_OBJ
    kernel = args[1] if len(args) > 1 else DEFAULT_KERNEL
    name, insns = kernel_sass(obj, kernel)
    (lo, hi), body = loop_body(insns)
    if by_callsite:
        print('kernel %s' % name)
        print_callsites(obj, name, lo, hi)
        return
    ops = collections.Counter(op.split('.')[0] for _, op, _ in body)
    dfma3r = sum(1 for _, op, args in body
                 if op.split('.')[0] == 'DFMA' and all(REG.match(a.strip()) for a in args.split(',')[1:]))
    print('kernel %s' % name)
    print('loop 0x%x..0x%x: %d instructions' % (lo, hi, len(body)))
    print('  FP64 (%s): %d' % ('/'.join(FP64), sum(ops[o] for o in FP64)))
    print('  DFMA with three R sources: %d' % dfma3r)
    for o in ('DFMA', 'DMUL', 'DADD', 'DSETP', 'FSEL', 'IMAD', 'MOV', 'LDC', 'LDCU', 'UMOV', 'MUFU'):
        print('  %-6s %d' % (o, ops[o]))
    print('all opcodes:', ' '.join('%s=%d' % kv for kv in ops.most_common()))


if __name__ == '__main__':
    main()
