"""CPU: the mbarrier, TMA, bulk-group and tcgen05 instructions are issued through the wrappers of csrc/tcgen05.cuh only.
A kernel file that spells one of them in its own inline PTX grows a private copy of that layer, and copies drift."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ladder-vae-pytorch_b200", "csrc")
WRAPPED = re.compile(r"mbarrier\.|tcgen05\.|cp\.async\.bulk|cp\.reduce\.async\.bulk")


def asm_templates(path):
    """(line number, instruction text) of every asm statement in a source file."""
    src = open(path, encoding="utf-8").read()
    for m in re.finditer(r"\basm\s*(?:volatile\s*)?\(", src):
        depth, i, text, in_template = 1, m.end(), [], True
        while depth:                                   # up to the closing parenthesis, skipping string contents
            c = src[i]
            if c == '"':
                j = i + 1
                while src[j] != '"':
                    j += 2 if src[j] == "\\" else 1
                if in_template:
                    text.append(src[i + 1:j])
                i = j
            elif c == ":" and depth == 1:              # operands and clobbers follow the instruction template
                in_template = False
            elif c == "(":
                depth += 1
            elif c == ")":
                depth -= 1
            i += 1
        yield src.count("\n", 0, m.start()) + 1, "".join(text)


def test_no_private_tcgen05_ptx_in_kernel_files():
    hits = ["%s:%d %s" % (os.path.basename(p), n, t.strip())
            for p in sorted(glob.glob(os.path.join(CSRC, "*.cu"))) for n, t in asm_templates(p) if WRAPPED.search(t)]
    assert not hits, "wrap these in csrc/tcgen05.cuh: %s" % hits


def test_scan_sees_the_header_wrappers():
    found = {WRAPPED.search(t).group(0) for _, t in asm_templates(os.path.join(CSRC, "tcgen05.cuh")) if WRAPPED.search(t)}
    assert found == {"mbarrier.", "tcgen05.", "cp.async.bulk", "cp.reduce.async.bulk"}
