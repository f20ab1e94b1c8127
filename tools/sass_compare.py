r"""Compare the machine code of two builds of libd3pm_b200.so, kernel by kernel.

    python tools/sass_compare.py OLD.so NEW.so [--context 3] [--rename PATTERN=REPLACEMENT ...]

Runs `cuobjdump -sass` on both libraries, splits each listing at its `Function :` lines and compares the kernels by
mangled name.  Reports the kernels that exist in only one build, the number that are byte-identical, and for each kernel
that differs a diff of its instructions, plus whether every change lies in the kernel's set-up, i.e. before its first
CTA-wide barrier (`__syncthreads()`, BAR.SYNC 0x0).  In that diff the encodings are dropped and the code addresses
inside instructions (branch targets, return addresses) are rewritten relative to the instruction, so code that merely
moved after an inserted or removed instruction compares equal.  Addresses shown are those of NEW.so.
--rename applies a regular-expression substitution to the kernel names of OLD.so before they are matched, for a kernel
whose mangled name changed while its code should not, e.g. a template that gained a parameter with a default value
(`--rename 'train_stream_kernelILi(\d)ELb(\d)EE=train_stream_kernelILi\1ELb\2ELi0EE'`).
Exit status 0 when every kernel is present in both builds and identical, 1 otherwise.
"""
import argparse
import difflib
import re
import subprocess
import sys

_FUNC = re.compile(r"^\s*Function : (\S+)\s*$")
_INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
_HEX = re.compile(r"\b0x([0-9a-f]+)\b")
_TARGET_OPS = ("BRA", "BSSY", "CALL", "JMP", "WARPSYNC")  # the hex operand is an absolute code address
_CTA_BARRIER = re.compile(r"^BAR\.SYNC(\.DEFER_BLOCKING)? 0x0$")


def functions(lib):
    """{mangled name: listing text} of every kernel in `lib`."""
    out = subprocess.run(["cuobjdump", "-sass", lib], check=True, capture_output=True, text=True).stdout
    funcs, name, lines = {}, None, []
    for line in out.splitlines():
        m = _FUNC.match(line)
        if m:
            if name is not None:
                funcs[name] = "\n".join(lines)
            name, lines = m.group(1), []
        elif name is not None:
            if line.startswith("Fatbin ") or line.strip().startswith("....."):
                funcs[name] = "\n".join(lines)
                name, lines = None, []
            else:
                lines.append(line)
    if name is not None:
        funcs[name] = "\n".join(lines)
    return funcs


def _relative(insn, addr):
    return _HEX.sub(lambda t: "%+d" % (int(t.group(1), 16) - addr), insn)


def instructions(text):
    """[(address, instruction)] without encodings, code addresses relative, trailing alignment NOPs dropped."""
    insns = []
    for line in text.splitlines():
        m = _INSN.match(line)
        if not m:
            continue
        addr, insn = int(m.group(1), 16), m.group(2)
        op = (insn.split()[1] if insn.startswith("@") else insn.split()[0]).split(".")[0]
        if op in _TARGET_OPS:
            insn = _relative(insn, addr)
        if op == "CALL":  # the MOV shortly before that loads the return address (the instruction after the call)
            for k in range(len(insns) - 1, max(-1, len(insns) - 9), -1):
                at, prev = insns[k]
                if prev.startswith("MOV ") and prev.endswith(f", {addr + 16:#x}"):
                    insns[k] = (at, _relative(prev, at))
                    break
        insns.append((addr, insn))
    while insns and insns[-1][1] == "NOP":
        insns.pop()
    return insns


def first_cta_barrier(insns):
    return next((i for i, (_, insn) in enumerate(insns) if _CTA_BARRIER.match(insn)), len(insns))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--context", type=int, default=3, help="unchanged instructions shown around each change")
    ap.add_argument("--rename", action="append", default=[], metavar="PATTERN=REPLACEMENT",
                    help="re.sub applied to the kernel names of OLD before matching (repeatable)")
    a = ap.parse_args()
    old, new = functions(a.old), functions(a.new)
    for rule in a.rename:
        pattern, _, replacement = rule.partition("=")
        old = {re.sub(pattern, replacement, name): text for name, text in old.items()}
    only_old, only_new = sorted(set(old) - set(new)), sorted(set(new) - set(old))
    common = sorted(set(old) & set(new))
    differ = [f for f in common if old[f] != new[f]]
    print(f"kernels: {len(old)} in {a.old}, {len(new)} in {a.new}, {len(common)} in both")
    for f in only_old:
        print(f"  only in old: {f}")
    for f in only_new:
        print(f"  only in new: {f}")
    print(f"byte-identical: {len(common) - len(differ)}; different: {len(differ)}")
    for f in differ:
        io, inew = instructions(old[f]), instructions(new[f])
        sm = difflib.SequenceMatcher(a=[i for _, i in io], b=[i for _, i in inew], autojunk=False)
        changes = [op for op in sm.get_opcodes() if op[0] != "equal"]
        bo, bn = first_cta_barrier(io), first_cta_barrier(inew)
        in_setup = all(i2 <= bo and j2 <= bn for _, _, i2, _, j2 in changes)
        where = f"/*{inew[bn][0]:04x}*/" if bn < len(inew) else "(none)"
        print(f"\n== {f}: {len(io)} -> {len(inew)} instructions; first CTA barrier at {where}; "
              f"{'all changes before it' if in_setup else 'CHANGES AFTER IT'}")
        for group in sm.get_grouped_opcodes(a.context):
            for tag, i1, i2, j1, j2 in group:
                if tag == "equal":
                    for addr, insn in inew[j1:j2]:
                        print(f"   /*{addr:04x}*/   {insn}")
                    continue
                for _, insn in io[i1:i2]:
                    print(f"             - {insn}")
                for addr, insn in inew[j1:j2]:
                    print(f"   /*{addr:04x}*/ + {insn}")
            print("   ...")
    return 0 if not (only_old or only_new or differ) else 1


if __name__ == "__main__":
    sys.exit(main())
