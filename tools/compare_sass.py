"""Per-kernel SASS identity of two builds of the library: which kernels compile to the same instructions.

    python tools/compare_sass.py OLD.so NEW.so [--strip-last-arg NAME ...]

Runs ``cuobjdump -sass`` on both files, splits the listing per kernel and demangles the names.  Instruction addresses,
encoding words, comments and line information are dropped, so two kernels compare equal when their instruction text
is the same.  A kernel template that gained a trailing template argument keeps its old instantiations' names only once
that argument is removed: ``--strip-last-arg`` names such templates (default: step_tma_kernel and step_kernel), and a
trailing ``false`` argument of them is stripped from a NEW name that OLD lacks when OLD has the stripped name (so a
template that already had the argument in OLD is compared as it is) -- NEW's ``true`` instantiations stay distinct and
are reported as new.  Prints one line per kernel (identical / changed / new / removed) and a summary; exits 1 when a kernel
of OLD is changed or missing in NEW.
"""
import argparse
import os
import re
import shutil
import subprocess
import sys


def tool(name):
    found = shutil.which(name) or os.path.join("/usr/local/cuda/bin", name)
    if not os.path.exists(found):
        raise SystemExit(f"{name} not found")
    return found


def demangle(names):
    out = subprocess.run([tool("c++filt")], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return out.splitlines()


def kernels(path):
    """{demangled name: [normalised instruction lines]} of every kernel in the library's sm_100a code."""
    listing = subprocess.run([tool("cuobjdump"), "-sass", path], capture_output=True, text=True, check=True).stdout
    mangled, bodies, cur = [], [], None
    for line in listing.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            mangled.append(m.group(1))
            cur = []
            bodies.append(cur)
            continue
        if cur is None:
            continue
        text = re.sub(r"/\*.*?\*/", "", line)            # addresses and encoding words
        text = re.sub(r"//.*", "", text).strip()         # comments, line information
        if not text or text.startswith(".") or text.startswith("#"):
            continue
        cur.append(re.sub(r"\s+", " ", text))
    return dict(zip(demangle(mangled), bodies))


def strip_last_arg(name, templates):
    """``ns::tmpl<a, b, false>(args)`` -> ``ns::tmpl<a, b>(args)`` for the named templates."""
    for t in templates:
        m = re.match(r"(.*\b" + re.escape(t) + r"<)([^<>]*)(>.*)$", name)
        if m:
            args = [a.strip() for a in m.group(2).split(",")]
            if len(args) > 1 and args[-1] == "false":
                return m.group(1) + ", ".join(args[:-1]) + m.group(3)
    return name


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--strip-last-arg", nargs="*", default=["step_tma_kernel", "step_kernel"])
    args = ap.parse_args()
    old = kernels(args.old)
    new = {}
    for name, body in kernels(args.new).items():
        stripped = strip_last_arg(name, args.strip_last_arg)
        new[stripped if name not in old and stripped in old else name] = body
    status = {}
    for name in sorted(set(old) | set(new)):
        if name not in new:
            status[name] = "removed"
        elif name not in old:
            status[name] = "new"
        else:
            status[name] = "identical" if old[name] == new[name] else "changed"
    for name, s in status.items():
        n_old = len(old.get(name, ()))
        n_new = len(new.get(name, ()))
        print(f"{s:9s}  {n_old:6d} -> {n_new:6d} instructions  {name}")
    counts = {s: sum(1 for v in status.values() if v == s) for s in ("identical", "changed", "new", "removed")}
    print(f"\n{os.path.basename(args.old)} -> {os.path.basename(args.new)}: "
          + ", ".join(f"{v} {k}" for k, v in counts.items()) + f" (stripped trailing 'false' of: {', '.join(args.strip_last_arg)})")
    return 1 if counts["changed"] or counts["removed"] else 0


if __name__ == "__main__":
    sys.exit(main())
