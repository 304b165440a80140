"""Compare the machine code of two builds of one CUDA object, kernel by kernel:
   python tools/sass_compare.py OLD.o NEW.o [--pair OLD=NEW ...] [--diff N]

A kernel is named by its demangled name without the parameter list (k_gamma_rs, k_alloc_cat<true, 384>).  A kernel
that was renamed is paired with --pair OLD=NEW; the rest are paired by name.  The listings of `cuobjdump -sass` are
compared after stripping what a refactor may move without changing the code: the symbol names, the instruction
addresses and encodings (branch targets become offsets from the branch), and the parameter offsets in constant bank 0
(c[0x0][...]), which change with a kernel's parameter list.  The registers, stack, local and shared memory of
`cuobjdump -res-usage` must match as well.  Prints one line per kernel (--diff N: also the first N differing lines) and
exits 1 if any kernel differs or has no partner."""
import argparse, difflib, os, re, subprocess, sys

CUDA = os.environ.get('CUDA_HOME', '/usr/local/cuda')
FUNC = re.compile(r'^\s*Function : (\S+)')
INSN = re.compile(r'^\s*/\*([0-9a-f]{4,})\*/\s*(.*?)\s*;')
TARGET = re.compile(r'^(?:@!?\w+\s+)?(?:BRA|BRX|JMP|JMX|CALL|BSSY|BREAK|SSY|PBK|PCNT)\b')
RES = re.compile(r'(REG|STACK|SHARED|LOCAL|CONSTANT\[0\]):(\d+)')


def tool(name, *args):
    return subprocess.run([os.path.join(CUDA, 'bin', name), *args], check=True, capture_output=True, text=True).stdout


def short_names(mangled):
    """mangled symbol -> demangled name without its parameter list"""
    out = {}
    for m, d in zip(mangled, tool('cu++filt', *mangled).splitlines()):
        d = d.strip()
        if d.endswith(')'):  # cut the parameter list: the last parenthesised group
            depth = 0
            for i in range(len(d) - 1, -1, -1):
                depth += d[i] == ')'
                depth -= d[i] == '('
                if depth == 0:
                    d = d[:i]
                    break
        d = re.sub(r'^void ', '', d)
        d = re.sub(r'\(bool\)0', 'false', re.sub(r'\(bool\)1', 'true', d))
        out[m] = re.sub(r'\(int\)(-?\d+)', r'\1', d)
    return out


def normalise(insns):
    """[(address, text)] of one kernel -> [text]: code addresses (branch targets, and the return addresses that a MOV
    hands to a CALL) become offsets in instructions from the instruction that holds them"""
    returns = {a + 16 for a, t in insns if re.match(r'^(?:@!?\w+\s+)?CALL\b', t)}
    out = []
    for addr, text in insns:
        text = re.sub(r'c\[0x0\]\[0x[0-9a-f]+\]', 'c[0x0][.]', text)
        m = re.search(r'\b0x([0-9a-f]+)$', text)
        if m and (TARGET.match(text) or (text.startswith('MOV ') and int(m.group(1), 16) in returns)):
            text = text[:m.start()] + '.%+d' % ((int(m.group(1), 16) - addr) // 16)
        out.append(re.sub(r'\s+', ' ', text))
    return out


def listings(obj):
    kernels, cur = {}, None
    for line in tool('cuobjdump', '-sass', obj).splitlines():
        f = FUNC.match(line)
        if f:
            cur = kernels.setdefault(f.group(1), [])
            continue
        i = INSN.match(line)
        if i and cur is not None:
            cur.append((int(i.group(1), 16), i.group(2)))
    res, cur = {}, None
    for line in tool('cuobjdump', '-res-usage', obj).splitlines():
        f = re.match(r'^\s*Function (\S+):', line)
        if f:
            cur = f.group(1)
        elif cur and 'REG:' in line:
            res[cur] = dict((k, int(v)) for k, v in RES.findall(line))
    names = short_names(sorted(kernels))
    return {names[m]: (normalise(kernels[m]), res.get(m, {})) for m in kernels}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('old')
    ap.add_argument('new')
    ap.add_argument('--pair', action='append', default=[], metavar='OLD=NEW')
    ap.add_argument('--diff', type=int, default=0, metavar='N')
    args = ap.parse_args()
    old, new = listings(args.old), listings(args.new)
    pairs = dict(p.split('=', 1) for p in args.pair)
    bad = 0
    for o in sorted(old):
        n = pairs.get(o, o)
        label = o if n == o else '%s -> %s' % (o, n)
        if n not in new:
            print('%-44s missing in %s' % (label, args.new))
            bad += 1
            continue
        (ia, ra), (ib, rb) = old[o], new[n]
        keys = ('REG', 'STACK', 'SHARED', 'LOCAL')
        res = ' '.join('%s %d' % (k, ra.get(k, -1)) for k in keys)
        same_res = all(ra.get(k) == rb.get(k) for k in keys)
        if not same_res:
            res = ' '.join('%s %d/%d' % (k, ra.get(k, -1), rb.get(k, -1)) for k in keys)
        params = '' if ra.get('CONSTANT[0]') == rb.get('CONSTANT[0]') else \
            '  param bank %d -> %d bytes' % (ra.get('CONSTANT[0]', -1), rb.get('CONSTANT[0]', -1))
        if ia == ib and same_res:
            print('%-44s same     %5d instructions  %s%s' % (label, len(ia), res, params))
            continue
        bad += 1
        delta = [l for l in difflib.unified_diff(ia, ib, lineterm='', n=0) if l[:1] in '+-' and l[:3] not in ('---', '+++')]
        print('%-44s DIFFERS  %5d -> %d instructions, %d lines differ  %s%s' % (label, len(ia), len(ib), len(delta), res, params))
        for l in delta[:args.diff]:
            print('    ' + l)
    for n in sorted(set(new) - {pairs.get(o, o) for o in old}):
        print('%-44s new in %s only' % (n, args.new))
        bad += 1
    return 1 if bad else 0


if __name__ == '__main__':
    sys.exit(main())
