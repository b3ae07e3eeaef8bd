"""Compares the SASS of the megakernel of two source trees, ignoring symbol names.

    python tools/sass_compare.py OLD_TREE [NEW_TREE]      (NEW_TREE defaults to this repository)

Compiles csrc/megakernel.cu of both trees for sm_100a with the library's flags (no GPU needed), dumps the SASS with
cuobjdump and compares the instruction listings of RenderMega<DBG, BATCH> (RenderMega<DBG, BATCH, 1> in a tree with
the supersampled batch, RenderMega<DBG, BATCH, 1, false> in a tree with the accumulated batch) for DBG and BATCH = false
and true, and those of the supersampled batch, RenderMega<DBG, true, SS> (SS = 2, 4, 8), wherever the old tree has it.
A tree from before the batch form only has the single-view kernel, RenderMega<DBG>, which is then compared with
BATCH = false alone.  Also prints ptxas' registers / stack / spill figures of every RenderMega instantiation, the
supersampled (SS = 2, 4, 8) and accumulating (ACC = true) ones included.  Exit status 0 when the listings are
identical.
"""
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mythtracer_b200.build import NVCC_FLAGS  # noqa: E402


def _compile(tree, out_dir):
    cubin = os.path.join(out_dir, "mega.cubin")
    nvcc = os.environ.get("NVCC", "nvcc")
    res = subprocess.run([nvcc] + NVCC_FLAGS + ["-Xptxas", "-v", "-I", os.path.join(tree, "include"), "-I",
                                                os.path.join(tree, "mythtracer_b200", "csrc"), "-cubin", "-o", cubin,
                                                os.path.join(tree, "mythtracer_b200", "csrc", "megakernel.cu")],
                         capture_output=True, text=True, check=True)
    sass = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    return res.stderr, sass


def _ptxas_figures(log):
    out = {}
    for m in re.finditer(r"Function properties for (\S*RenderMega\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                         r"(\d+) bytes spill loads\n.*?Used (\d+) registers", log):
        out[m.group(1)] = dict(stack=int(m.group(2)), spill_stores=int(m.group(3)), spill_loads=int(m.group(4)), registers=int(m.group(5)))
    return out


def _functions(sass):
    """{mangled name: [instruction text]} without addresses and encodings."""
    funcs = {}
    for block in sass.split("Function : ")[1:]:
        name, body = block.split("\n", 1)
        funcs[name.strip()] = [m.group(1).strip() for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;", body)]
    return funcs


def _instantiation(funcs, dbg, batch, ss=1):
    """(name, code) of RenderMega<dbg, batch, ss> (<dbg, batch> for ss = 1 without the SS parameter, <..., false> with
    the ACC parameter; <dbg> stands for <dbg, false>), or None."""
    if ss == 1:
        patterns = [r"RenderMegaILb%dELb%dE(Li1E(Lb0E)?)?EEv" % (dbg, batch)] + ([r"RenderMegaILb%dEEEv" % dbg] if not batch else [])
    else:
        patterns = [r"RenderMegaILb%dELb%dELi%dE(Lb0E)?EEv" % (dbg, batch, ss)]
    for name, code in funcs.items():
        if any(re.search(p, name) for p in patterns):
            return name, code
    return None


def main():
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    old_tree, new_tree = sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else ROOT
    same = True
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "old"))
        os.makedirs(os.path.join(tmp, "new"))
        old_log, old_sass = _compile(old_tree, os.path.join(tmp, "old"))
        new_log, new_sass = _compile(new_tree, os.path.join(tmp, "new"))
    for label, log in (("old", old_log), ("new", new_log)):
        for name, fig in _ptxas_figures(log).items():
            print("%s %s %s" % (label, re.search(r"RenderMega\w*?E(?=EvN)", name).group(0), fig))
    old_f, new_f = _functions(old_sass), _functions(new_sass)
    for batch, ss in ((0, 1), (1, 1), (1, 2), (1, 4), (1, 8)):
        for dbg in (0, 1):
            old, new = _instantiation(old_f, dbg, batch, ss), _instantiation(new_f, dbg, batch, ss)
            if new is None:
                raise SystemExit("no RenderMega<%d, %d, %d> in the listing of %s" % (dbg, batch, ss, new_tree))
            if old is None:
                if not batch:
                    raise SystemExit("no single-view RenderMega<%d> in the listing of %s" % (dbg, old_tree))
                print("RenderMega<DBG=%d, BATCH=1, SS=%d>: not in %s" % (dbg, ss, old_tree))
                continue
            (on, oc), (nn, nc) = old, new
            equal = oc == nc
            same &= equal
            print("RenderMega<DBG=%d, BATCH=%d, SS=%d>: %d vs %d instructions, %s" % (dbg, batch, ss, len(oc), len(nc),
                                                                                    "identical" if equal else "DIFFERENT"))
            if not equal:
                for i, (a, b) in enumerate(zip(oc, nc)):
                    if a != b:
                        print("  first difference at instruction %d: %s | %s" % (i, a, b))
                        break
    sys.exit(0 if same else 1)


if __name__ == "__main__":
    main()
