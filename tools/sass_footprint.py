"""Static footprint of a kernel's interior-point loop in SASS (runs without a GPU).

Given a built libbnmpc.so or object file, extract the sm_100a cubin(s) with `cuobjdump -xelf all`, disassemble them with
`nvdisasm -g` (the library is built with -lineinfo) and, for one kernel, report the byte span of the interior-point loop:
the block of instructions attributed to the source lines of `Solver::residual_pass` ... `Solver::qp_ipm` in
bnmpc_core.cuh.  The line range is read from the header itself, so it follows edits.  Inside the span: instruction count,
opcode mix and the source lines that hold the most instructions (every file, so inlined helpers show up where they sit).

    python tools/sass_footprint.py drone_attitude_control_b200/lib/libbnmpc.so
    python tools/sass_footprint.py build/csrc/model_jerk.o --kernel 'k_loop_step<Model_jerk, double, 1>' --json

Why it matters: a multi-step launch lets the warps of an SM drift apart, and each then fetches the loop on its own; a
loop larger than the instruction cache turns into `no-instruction` stalls (profiles/README.md).
"""
import argparse
import bisect
import collections
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CORE = os.path.join(ROOT, 'drone_attitude_control_b200', 'csrc', 'bnmpc_core.cuh')
INSN_BYTES = 16
# a run of this many bytes without an attributed instruction ends a block (the loop is one block; out-of-line slow paths
# placed elsewhere in the kernel are reported separately)
GAP_BYTES = 2048


def tool(name):
    p = shutil.which(name) or os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'bin', name)
    if not os.path.exists(p):
        raise SystemExit(f'{name} not found (CUDA toolkit bin directory on PATH or CUDA_HOME)')
    return p


def loop_lines(core=CORE, first='residual_pass', last='qp_ipm'):
    """[start, end] source lines of bnmpc_core.cuh from the definition of `first` to the closing brace of `last`."""
    src = open(core).read().split('\n')
    def defline(name):
        pat = re.compile(r'^\s*BN_HD\s+[\w:<>,\s\*&]+?\b' + name + r'\s*\(')
        for i, l in enumerate(src):
            if pat.match(l):
                return i
        raise SystemExit(f'no definition of {name} in {core}')
    a, b = defline(first), defline(last)
    depth, seen = 0, False
    for i in range(b, len(src)):
        depth += src[i].count('{') - src[i].count('}')
        seen = seen or '{' in src[i]
        if seen and depth == 0:
            return a + 1, i + 1
    raise SystemExit(f'unbalanced braces after {last} in {core}')


def demangle(names):
    if not names:
        return {}
    out = subprocess.run([tool('cu++filt')], input='\n'.join(names), capture_output=True, text=True, check=True).stdout
    return dict(zip(names, out.strip('\n').split('\n')))


def norm(s):
    """spelling-independent kernel name: no blanks, no namespace qualifiers, no '(int)' casts of template arguments"""
    return re.sub(r'\w+::|\(int\)|\s+', '', s)


def kernel_key(demangled):
    """'bnmpc::k_loop_step<Model_force, double, 1>(...)' -> 'k_loop_step<Model_force,double,1>'"""
    d = demangled
    if d.startswith('void '):
        d = d[5:]
    depth = 0
    for i, ch in enumerate(d):           # cut the argument list: the first '(' outside template brackets
        if ch == '<': depth += 1
        elif ch == '>': depth -= 1
        elif ch == '(' and depth == 0:
            d = d[:i]
            break
    t = d.find('<') if '<' in d else len(d)
    return norm(d[:t].split('::')[-1] + d[t:])


def disassemble(binary, work):
    """{mangled kernel name: [(address, opcode, file, line)]} over every cubin inside `binary`."""
    if binary.endswith('.cubin'):
        cubins = [binary]
    else:
        subprocess.run([tool('cuobjdump'), '-xelf', 'all', os.path.abspath(binary)], cwd=work, check=True,
                       capture_output=True)
        cubins = [os.path.join(work, f) for f in sorted(os.listdir(work)) if f.endswith('.cubin')]
    if not cubins:
        raise SystemExit(f'no cubin in {binary}')
    sec = re.compile(r'^\s*\.section\s+\.text\.([^,\s]+)')
    loc = re.compile(r'^\s*//## File "([^"]+)", line (\d+)')
    ins = re.compile(r'^\s*/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)')
    kernels = {}
    for cb in cubins:
        text = subprocess.run([tool('nvdisasm'), '-g', '-c', cb], capture_output=True, text=True, check=True).stdout
        cur, f, ln = None, None, None
        for l in text.split('\n'):
            m = sec.match(l)
            if m:
                cur = kernels.setdefault(m.group(1), []); f, ln = None, None
                continue
            m = loc.match(l)
            if m:
                f, ln = os.path.basename(m.group(1)), int(m.group(2))
                continue
            m = ins.match(l)
            if m and cur is not None:
                cur.append((int(m.group(1), 16), m.group(2), f, ln))
    return kernels


def footprint(insns, lines, core_file=os.path.basename(CORE)):
    lo, hi = lines
    hits = [a for a, _, f, ln in insns if f == core_file and ln is not None and lo <= ln <= hi]
    if not hits:
        return None
    blocks, start, prev = [], hits[0], hits[0]
    for a in hits[1:]:
        if a - prev > GAP_BYTES:
            blocks.append((start, prev)); start = a
        prev = a
    blocks.append((start, prev))
    def count(b): return sum(1 for a in hits if b[0] <= a <= b[1])
    main = max(blocks, key=count)
    span = [x for x in insns if main[0] <= x[0] <= main[1]]
    ops = collections.Counter(op.split('.')[0] for _, op, _, _ in span)
    src = collections.Counter(f'{f}:{ln}' if f else '?' for _, _, f, ln in span)
    return {
        'span': [main[0], main[1] + INSN_BYTES],
        'bytes': main[1] + INSN_BYTES - main[0],
        'instructions': len(span),
        'kernel_instructions': len(insns),
        'attributed_to_loop_lines': count(main),
        'outside_blocks': [[b[0], b[1] + INSN_BYTES, count(b)] for b in blocks if b != main],
        'opcodes': ops.most_common(),
        'source_lines': src.most_common(),
        'loop_lines': [lo, hi],
    }


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('binary', help='libbnmpc.so, an object file of csrc/ or a cubin')
    ap.add_argument('--kernel', default='k_loop_step<Model_force, double, 1>',
                    help='kernel name as in the source, template arguments included (default: %(default)s)')
    ap.add_argument('--core', default=CORE, help='the bnmpc_core.cuh the binary was built from (default: this tree)')
    ap.add_argument('--top', type=int, default=25, help='opcodes / source lines to list')
    ap.add_argument('--json', action='store_true', help='print one JSON object instead of the table')
    ap.add_argument('--list', action='store_true', help='list the kernels in the binary and exit')
    a = ap.parse_args(argv)
    with tempfile.TemporaryDirectory() as work:
        kernels = disassemble(a.binary, work)
    names = demangle(sorted(kernels))
    if a.list:
        for m in sorted(kernels):
            print(f'{len(kernels[m]) * INSN_BYTES:8d} B  {names.get(m, m)}')
        return 0
    want = norm(a.kernel)
    match = [m for m in kernels if kernel_key(names.get(m, m)) == want]
    if len(match) != 1:
        print(f'kernel {a.kernel!r}: {len(match)} matches; --list shows the kernels', file=sys.stderr)
        return 2
    lines = loop_lines(a.core)
    fp = footprint(kernels[match[0]], lines)
    if fp is None:
        print(f'no instruction of {a.kernel} is attributed to bnmpc_core.cuh:{lines[0]}-{lines[1]} '
              '(built without -lineinfo?)', file=sys.stderr)
        return 2
    fp['kernel'] = a.kernel
    if a.json:
        print(json.dumps(fp))
        return 0
    print(f'{a.kernel}: {fp["kernel_instructions"]} instructions ({fp["kernel_instructions"] * INSN_BYTES / 1024:.1f} KB)')
    print(f'interior-point loop (bnmpc_core.cuh:{lines[0]}-{lines[1]}, residual_pass ... qp_ipm): '
          f'0x{fp["span"][0]:x}-0x{fp["span"][1]:x} = {fp["bytes"]} B ({fp["bytes"] / 1024:.1f} KB), '
          f'{fp["instructions"]} instructions, {fp["attributed_to_loop_lines"]} of them on the loop lines')
    for b in fp['outside_blocks']:
        print(f'  outside the span: 0x{b[0]:x}-0x{b[1]:x}, {b[2]} loop-line instructions')
    print('opcodes: ' + ', '.join(f'{o} {c}' for o, c in fp['opcodes'][:a.top]))
    print('source lines inside the span:')
    for s, c in fp['source_lines'][:a.top]:
        print(f'  {c:5d}  {s}')
    return 0


if __name__ == '__main__':
    sys.exit(main())
