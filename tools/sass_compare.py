"""Compares the SASS of every kernel of the megakernel and wavefront sources of two source trees.

    python tools/sass_compare.py OLD_TREE [NEW_TREE]      (NEW_TREE defaults to this repository)

Compiles csrc/megakernel.cu and csrc/wavefront.cu of both trees for sm_100a with the library's flags (no GPU needed),
dumps the SASS with cuobjdump and compares the instruction listings of every kernel by name.  Kernels are matched by
their demangled names: a mangled name contains a per-file hash of the anonymous namespace, which changes whenever the
file's content does.  Prints ptxas' registers / stack / spill figures of every kernel in both trees.  A kernel that
only the old tree has is listed as removed, one that only the new tree has as added; neither is a difference.  Exit
status 0 when every kernel of both trees has the same instruction listing and the same ptxas figures.
"""
import os
import re
import shutil
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mythtracer_b200.build import NVCC_FLAGS  # noqa: E402

SOURCES = ("megakernel.cu", "wavefront.cu")
NVCC = os.environ.get("NVCC", "nvcc")


def _compile(tree, src, out_dir):
    """(ptxas log, SASS listing) of csrc/<src> of `tree`, or None when the tree has no such file."""
    path = os.path.join(tree, "mythtracer_b200", "csrc", src)
    if not os.path.exists(path):
        return None
    cubin = os.path.join(out_dir, src + ".cubin")
    res = subprocess.run([NVCC] + NVCC_FLAGS + ["-Xptxas", "-v", "-I", os.path.join(tree, "include"), "-I",
                                                os.path.dirname(path), "-cubin", "-o", cubin, path],
                         capture_output=True, text=True, check=True)
    sass = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    return res.stderr, sass


def _demangle(names):
    filt = os.path.join(os.path.dirname(shutil.which(NVCC) or NVCC), "cu++filt")
    out = subprocess.run([filt if os.path.exists(filt) else "cu++filt"] + names, capture_output=True, text=True,
                         check=True).stdout.splitlines()
    return dict(zip(names, out))


def _short(demangled):
    """RenderMega<false, true, 8, false> for void mtb::<unnamed>::RenderMega<(bool)0, (bool)1, (int)8, (bool)0>(...)."""
    name = re.sub(r"\(bool\)([01])", lambda m: "true" if m.group(1) == "1" else "false", demangled).replace("(int)", "")
    return re.sub(r"^void |\(.*$", "", name).replace("mtb::<unnamed>::", "")


def _key(demangled):
    """The name a kernel is matched by: its short name, with RenderMega's trailing primary-ray parameters dropped while
    they are false (PANO, then LENS), so that RenderMega<a, b, c, d, e, false> of a tree with panoramas meets
    RenderMega<a, b, c, d, e> of one without, and RenderMega<a, b, c, d, false> meets RenderMega<a, b, c, d> of a tree
    without thin-lens views."""
    name = re.sub(r"^(RenderMega<[^,<>]+, [^,<>]+, [^,<>]+, [^,<>]+, [^,<>]+), false>$", r"\1>", _short(demangled))
    return re.sub(r"^(RenderMega<[^,<>]+, [^,<>]+, [^,<>]+, [^,<>]+), false>$", r"\1>", name)


def _kernels(log, sass):
    """{_key name: (ptxas figures, [instruction text])}: listings without addresses and encodings."""
    figures = {}
    for m in re.finditer(r"Compiling entry function '(\S+)'.*?\n.*?Function properties for \1\n\s*(\d+) bytes stack frame, "
                         r"(\d+) bytes spill stores, (\d+) bytes spill loads\n.*?Used (\d+) registers", log):
        figures[m.group(1)] = "%s registers, %s B stack, %s / %s B spill stores / loads" % (m.group(5), m.group(2), m.group(3),
                                                                                            m.group(4))
    code = {}
    for block in sass.split("Function : ")[1:]:
        name, body = block.split("\n", 1)
        code[name.strip()] = [m.group(1).strip() for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;", body)]
    missing = sorted(set(code) - set(figures))
    if missing:
        raise SystemExit("no ptxas figures for the kernel(s) %s" % ", ".join(missing))
    names = _demangle(sorted(code))
    return {_key(names[n]): (figures[n], c) for n, c in code.items()}


def main():
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    old_tree, new_tree = sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else ROOT
    jobs = [(tree, src) for src in SOURCES for tree in (old_tree, new_tree)]
    with tempfile.TemporaryDirectory() as tmp, ThreadPoolExecutor(len(jobs)) as pool:
        dirs = [os.path.join(tmp, str(i)) for i in range(len(jobs))]
        for d in dirs:
            os.makedirs(d)
        results = list(pool.map(lambda job, d: _compile(job[0], job[1], d), jobs, dirs))
    same = True
    for k, src in enumerate(SOURCES):
        old_res, new_res = results[2 * k], results[2 * k + 1]
        if new_res is None:
            raise SystemExit("no %s in %s" % (src, new_tree))
        old, new = _kernels(*old_res) if old_res else {}, _kernels(*new_res)
        print("%s:" % src)
        for name in sorted(set(old) | set(new)):
            if name not in new:
                print("  %s: removed (old: %s)" % (name, old[name][0]))
                continue
            if name not in old:
                print("  %s: added (new: %s)" % (name, new[name][0]))
                continue
            (of, oc), (nf, nc) = old[name], new[name]
            equal = oc == nc and of == nf
            same &= equal
            print("  %s: %d vs %d instructions, %s" % (name, len(oc), len(nc), "identical" if equal else "DIFFERENT"))
            print("    old: %s\n    new: %s" % (of, nf))
            if oc != nc:
                i = next((i for i, (a, b) in enumerate(zip(oc, nc)) if a != b), min(len(oc), len(nc)))
                print("    first difference at instruction %d: %s | %s" % (i, oc[i] if i < len(oc) else "(end)",
                                                                           nc[i] if i < len(nc) else "(end)"))
    sys.exit(0 if same else 1)


if __name__ == "__main__":
    main()
