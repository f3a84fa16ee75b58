"""The interior-point loop of the headline kernel stays small.

A multi-step launch lets the 16 warps of an SM drift apart, and each one then fetches the loop's instructions on its
own: a loop that outgrows the instruction cache turns into `no-instruction` stalls (DESIGN.md section 5).  This reads
the SASS of the built library (tools/sass_footprint.py: cuobjdump + nvdisasm, no GPU) and fails when the loop's byte
span grows past its budget, so a later change cannot push it back out of the cache unnoticed."""
import os
import shutil
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import sass_footprint as sf  # noqa: E402

LIB = os.path.join(ROOT, 'drone_attitude_control_b200', 'lib', 'libbnmpc.so')
KERNEL = 'k_loop_step<Model_force, double, 1>'
# bytes of SASS between the first and the last instruction of residual_pass ... qp_ipm in KERNEL (built as csrc/Makefile
# does, CUDA 12.9): 41 024 before the loop's bookkeeping was trimmed, 38 512 after
BUDGET = 39 * 1024


def cuda_tool(name):
    return shutil.which(name) or os.path.exists(os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'bin', name))


needs_build = pytest.mark.skipif(not os.path.exists(LIB) or not all(cuda_tool(t) for t in ('cuobjdump', 'nvdisasm', 'cu++filt')),
                                 reason='libbnmpc.so not built or CUDA binary utilities not installed')


def test_loop_lines_follow_the_source():
    lo, hi = sf.loop_lines()
    src = open(sf.CORE).read().split('\n')
    assert 'residual_pass(' in src[lo - 1]
    assert src[hi - 1].strip() == '}' and any('qp_ipm(' in l for l in src[lo - 1:hi])


def test_kernel_names_match_however_spelled():
    d = 'void bnmpc::k_loop_step<bnmpc::Model_force, double, (int)1>(bnmpc::Gs<T2>, bnmpc::Opts, bnmpc::LoopArgs, int *, int)'
    assert sf.kernel_key(d) == sf.norm(KERNEL)


@needs_build
def test_interior_point_loop_fits_its_budget():
    with __import__('tempfile').TemporaryDirectory() as work:
        kernels = sf.disassemble(LIB, work)
    names = sf.demangle(sorted(kernels))
    match = [m for m in kernels if sf.kernel_key(names[m]) == sf.norm(KERNEL)]
    assert len(match) == 1, 'kernel not found in libbnmpc.so'
    fp = sf.footprint(kernels[match[0]], sf.loop_lines())
    assert fp is not None, 'no line info in libbnmpc.so (csrc/Makefile builds with -lineinfo)'
    # the loop is one block: nearly all of its own instructions sit inside the span
    assert sum(b[2] for b in fp['outside_blocks']) <= 0.02 * fp['attributed_to_loop_lines']
    assert fp['bytes'] <= BUDGET, (f'interior-point loop of {KERNEL} is {fp["bytes"]} B, budget {BUDGET} B; '
                                   f'largest source lines: {fp["source_lines"][:10]}')
