"""CPU: the SASS of the frame kernels' FAST Binet loops (binet_trace_fast, lp_internal.cuh) stays at its
FP64 floor.  cuobjdump disassembles the built library; no GPU needed.

A FAST loop iteration is two trips of TRIP RK4 steps on ping-pong registers.  On the path that stays in the
loop it may hold only the RK4 steps' FP64 instructions and the bookkeeping the design needs: per trip, the
integer band test (TRIP high-word subtract / max, one compare, one branch) and, per iteration, the step
counter (one add, one compare; its branch is the second trip's).  Register copies, reconvergence barriers
and local memory there mean the compiler has re-introduced per-trip overhead: FP64 instructions hold the
issue port for two cycles each (DESIGN.md §4), so every extra instruction is paid on every trip."""
import re
import subprocess

import pytest

STEP_FP64 = {True: 14, False: 34}      # FP64 instructions of one RK4 step: FUSED (rk4_step_scaled), strict
FP64 = re.compile(r"^(DFMA|DADD|DMUL)\b")
KERNELS = {"lp_render_mirror_kernel": "_Z23lp_render_mirror_kernel", "lp_render_kernel": "_Z16lp_render_kernel"}
ELEMS = {"u8": "h", "f32": "f", "f64": "d"}
ARGS = "EEv9TraceArgs9RemapArgs11BinetConsts9CamConsts"


def _mangled(kernel, fused, elem, trip):
    return "%sILb%dELb1E%sLi4ELi%d%s" % (KERNELS[kernel], int(fused), ELEMS[elem], trip, ARGS)


CASES = [(k, f, e, t) for k in KERNELS for f in (True, False) for e in ELEMS for t in (2, 4)]


@pytest.fixture(scope="module")
def sass(native):
    names = [_mangled(*c) for c in CASES]
    out = subprocess.run(["cuobjdump", "-sass", "-fun", ",".join(names), native.LIB_PATH],
                         capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
            continue
        m = re.match(r"\s*/\*([0-9a-f]+)\*/\s+(.*?)\s*;", line)
        if m and name:
            funcs[name].append((int(m.group(1), 16), m.group(2).strip()))
    return funcs


def _opcode(text):
    return re.sub(r"^@!?U?P\w+\s+", "", text).split()[0]


def _innermost_loops(ins):
    """[first, back edge] address ranges of the loops that contain no other loop's back edge."""
    loops = []
    for addr, text in ins:
        m = re.match(r"(@!?U?P\w+\s+)?BRA(\.\w+)*\s+(!?U?P\w+,\s*)?0x([0-9a-f]+)$", text)
        if m and int(m.group(4), 16) <= addr:
            loops.append((int(m.group(4), 16), addr))
    return [l for l in loops if not any(o != l and l[0] <= o[0] and o[1] < l[1] for o in loops)]


def _main_loop(ins, fused):
    """The innermost loop with the most FP64 instructions among those of the step's kind (the strict step
    multiplies, DMUL; the FUSED one does not): its opcodes."""
    best = None
    for lo, hi in _innermost_loops(ins):
        ops = [_opcode(t) for a, t in ins if lo <= a <= hi]
        n = sum(1 for o in ops if FP64.match(o))
        if ("DMUL" in ops) == (not fused) and (best is None or n > best[0]):
            best = (n, ops, lo, hi)
    assert best is not None, "no loop of the step's kind"
    return best


def _violations(ins, fused, trip):
    n, ops, lo, hi = _main_loop(ins, fused)
    other = [o for o in ops if not FP64.match(o)]
    where = "loop 0x%x-0x%x" % (lo, hi)
    bad = []
    if n != STEP_FP64[fused] * 2 * trip:
        bad.append("%s: %d FP64 instructions, expected %d (two trips of %d steps)" % (where, n, STEP_FP64[fused] * 2 * trip, trip))
    if len(other) > 2 * (trip + 2) + 2:
        bad.append("%s: %d other instructions, at most %d: %s" % (where, len(other), 2 * (trip + 2) + 2, other))
    for what, pat in (("register copy", r"^(IMAD\.MOV|MOV)"), ("reconvergence", r"^(BSSY|BSYNC|BREAK|WARPSYNC)"),
                      ("local memory", r"^(STL|LDL)")):
        hits = [o for o in other if re.match(pat, o)]
        if hits:
            bad.append("%s: %s %s" % (where, what, hits))
    return bad


@pytest.mark.parametrize("kernel,fused,elem,trip", CASES)
def test_fast_loop_at_fp64_floor(sass, kernel, fused, elem, trip):
    ins = sass[_mangled(kernel, fused, elem, trip)]
    bad = _violations(ins, fused, trip)
    if fused:     # the strict re-trace of LP_TRACE_HYBRID inside the same kernel: binet_trace_fast<false, 2>
        bad += ["strict re-trace " + b for b in _violations(ins, False, 2)]
    assert not bad, "\n".join(bad)
