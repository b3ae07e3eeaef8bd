"""Register budget of the traversal kernels of a built library: registers, stack frame and local-memory instructions.

    python tools/reg_budget.py [LIB]      (a library or a cubin; default mythtracer_b200/libmythtracer_b200.so)

No GPU needed.  Extracts the cubins of LIB with cuobjdump, reads every RenderMega and WfQueue instantiation's registers
and stack frame (cuobjdump -res-usage) and its SASS with line information (nvdisasm -gi; the library is built with
-lineinfo), and counts the local-memory instructions (LDL / STL) of the whole kernel and of two loops of TraceFast
(device_core.cuh):
  node  the node loop: the innermost loop around the two 256-bit loads of a scene-BVH node;
  slot  the per-slot leaf loop: the innermost loop around the 256-bit loads of a triangle record (TestSlotFast).
A loop is the address range from the target of a backward branch to that branch.  Each count is split into fixed
slots ([R1 + offset]: spill slots and the fixed-offset per-pixel state) and indexed accesses (a computed address: the
traversal stack's push and pop).  Prints one line per kernel; exit status 1 when a kernel has no such loop.
"""
import os
import re
import shutil
import subprocess
import sys
import tempfile
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = re.compile(r"^(RenderMega|WfQueue)<")
# the inline asm of the two loads, found through the SASS line information: an instruction carries the LAST line of a
# statement, and the node load's statement spans three (the source files must be where they were compiled)
NODE_LOAD, SLOT_LOAD = "ld.global.nc.v8.f32", "ld.global.nc.v4.f64"


_sources = {}


def _source_line(path, n):
    """Line n of the source file the line information names ("" when it cannot be read)."""
    if path not in _sources:
        try:
            with open(path) as f:
                _sources[path] = f.read().splitlines()
        except OSError:
            _sources[path] = []
    lines = _sources[path]
    return lines[n - 1] if 0 < n <= len(lines) else ""


def _short(mangled):
    name = subprocess.run(["cu++filt", mangled], capture_output=True, text=True, check=True).stdout.strip()
    name = re.sub(r"\(bool\)([01])", lambda m: "true" if m.group(1) == "1" else "false", name).replace("(int)", "")
    return re.sub(r"^void |\(.*$", "", name).replace("mtb::<unnamed>::", "")


def _parse(listing):
    """[(address, instruction text, set of (file, line) in its inline chain)] and {label: instruction index}."""
    code, labels, chain, pending = [], {}, set(), []
    for line in listing.splitlines():
        m = re.match(r'\s*//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?', line)
        if m:
            if not pending:
                chain = set()
            pending.append(line)
            chain.add((m.group(1), int(m.group(2))))
            if m.group(3):
                chain.add((m.group(3), int(m.group(4))))
            continue
        m = re.match(r"\s*(\.L_x_\d+):", line)
        if m:
            labels[m.group(1)] = len(code)
            continue
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s*(.*?)\s*;", line)
        if m:
            code.append((int(m.group(1), 16), m.group(2), chain))
            pending = []
    return code, labels


def _loop(code, labels, anchor):
    """(first, last) instruction index of the innermost backward-branch range around instruction `anchor`."""
    best = None
    for i, (_, text, _) in enumerate(code):
        m = re.search(r"\bBRA\b.*`\((\.L_x_\d+)\)", text)
        if m and m.group(1) in labels and labels[m.group(1)] <= anchor <= i:
            if best is None or i - labels[m.group(1)] < best[1] - best[0]:
                best = (labels[m.group(1)], i)
    return best


def _local(instrs):
    c = Counter()
    for text in instrs:
        m = re.search(r"\b(LDL|STL)\b[^\[]*\[([^\]]+)\]", text)
        if m:
            c[m.group(1) + ("" if re.fullmatch(r"R1(\+0x[0-9a-f]+)?", m.group(2).replace(" ", "")) else "[idx]")] += 1
    return c


def _fmt(c):
    return "LDL %d STL %d, indexed LDL %d STL %d" % (c["LDL"], c["STL"], c["LDL[idx]"], c["STL[idx]"])


def report(lib):
    ok = True
    with tempfile.TemporaryDirectory() as tmp:
        if lib.endswith(".cubin"):
            shutil.copy(lib, tmp)
        else:
            subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=tmp, capture_output=True, check=True)
        for cubin in sorted(f for f in os.listdir(tmp) if f.endswith(".cubin")):
            path = os.path.join(tmp, cubin)
            usage = subprocess.run(["cuobjdump", "-res-usage", path], capture_output=True, text=True, check=True).stdout
            res = {f: (r, s) for f, r, s in re.findall(r"Function (\S+):\n\s*REG:(\d+) STACK:(\d+)", usage)}
            names = [f for f in res if KERNELS.match(_short(f))]
            if not names:
                continue
            sass = subprocess.run(["nvdisasm", "-gi", path], capture_output=True, text=True, check=True).stdout
            sections = dict(re.findall(r"\.section\s+\.text\.(\S+?),\"ax\"[^\n]*\n(.*?)(?=\n\s*\.section|\Z)", sass, re.S))
            for f in sorted(names, key=_short):
                code, labels = _parse(sections[f])
                line = "%s: %s registers, %s B stack, kernel %s" % (_short(f), res[f][0], res[f][1], _fmt(_local(t for _, t, _ in code)))
                for tag, asm in (("node", NODE_LOAD), ("slot", SLOT_LOAD)):
                    at = next((i for i, (_, t, ch) in enumerate(code) if ".256" in t and any(asm in _source_line(f_, n - k) for f_, n in ch for k in range(3))), None)
                    rng = _loop(code, labels, at) if at is not None else None
                    if rng is None:
                        ok = False
                        line += "; %s loop: not found" % tag
                        continue
                    line += "; %s loop (%d instructions): %s" % (tag, rng[1] - rng[0] + 1, _fmt(_local(t for _, t, _ in code[rng[0]:rng[1] + 1])))
                print(line)
    return ok


if __name__ == "__main__":
    sys.exit(0 if report(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "mythtracer_b200", "libmythtracer_b200.so")) else 1)
