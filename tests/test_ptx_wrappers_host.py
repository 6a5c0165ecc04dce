"""CPU: the mbarrier, cp.async, TMA, tcgen05, elect.sync and async-proxy fence PTX is spelled in csrc/ptx.cuh only.
Every other kernel source calls its wrappers, so the instruction forms (operands, clobbers, predicates) cannot drift
between copies."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "unnamed-rust-sdr_b200", "csrc")
FAMILIES = ("mbarrier.", "cp.async", "tcgen05.", "elect.sync", "fence.proxy.async", "fence.mbarrier_init")


def asm_strings(src):
    """The concatenated string literals of every asm statement in C++ source `src`; comments are skipped."""
    masked, lits = [], []  # masked: src with comments and string contents blanked; lits: (offset, contents)
    i, n = 0, len(src)
    while i < n:
        c = src[i]
        if src.startswith("//", i):
            j = src.find("\n", i)
            j = n if j < 0 else j
        elif src.startswith("/*", i):
            j = src.find("*/", i + 2) + 2
        elif c in "\"'":
            j = i + 1
            while src[j] != c:
                j += 2 if src[j] == "\\" else 1
            j += 1
            if c == '"':
                lits.append((i, src[i + 1:j - 1]))
        else:
            masked.append(c)
            i += 1
            continue
        masked.append(" " * (j - i))
        i = j
    masked = "".join(masked)
    out = []
    for m in re.finditer(r"\basm\s*(?:volatile\b|__volatile__\b)?\s*\(", masked):
        depth, j = 1, m.end()
        while depth:
            depth += {"(": 1, ")": -1}.get(masked[j], 0)
            j += 1
        out.append("".join(s for k, s in lits if m.end() <= k < j))
    return out


def families_in(path):
    found = set()
    for s in asm_strings(open(path).read()):
        found.update(f for f in FAMILIES if f in s)
    return found


def test_scanner_reads_asm_strings_only():
    src = ('// cp.async.wait_group in prose\n/* tcgen05.mma */ const char *s = "elect.sync";\n'
           'asm volatile("{\\n mbarrier.try_wait %0;\\n}" : "=r"(x) : "r"(f("(")));\n')
    assert asm_strings(src) == ["{\\n mbarrier.try_wait %0;\\n}=rr("]


def test_ptx_families_are_spelled_in_ptx_cuh_only():
    assert families_in(os.path.join(CSRC, "ptx.cuh")) == set(FAMILIES)
    stray = {}
    for path in sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh"))):
        if os.path.basename(path) != "ptx.cuh":
            found = families_in(path)
            if found:
                stray[os.path.basename(path)] = sorted(found)
    assert not stray, f"PTX outside ptx.cuh (call its wrappers instead): {stray}"
