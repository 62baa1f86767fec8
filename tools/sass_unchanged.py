#!/usr/bin/env python3
"""Check that every kernel of an older build of libmarlsc_b200.so compiles to the same machine code in a newer one.

    python tools/sass_unchanged.py OLD.so NEW.so

Runs ``cuobjdump -sass`` and ``cuobjdump -res-usage`` on both libraries (no GPU needed), demangles the kernel names
and identifies a kernel by its qualified name and template arguments (parameter lists are left out: a kernel may gain
a trailing parameter that its old instantiations never read). A kernel template that gained a trailing ``bool`` template
argument, default ``false``, is matched through that argument: ``k<1, 2, false>`` of the new build stands for ``k<1, 2>``
of the old one (``k<false>`` for ``k``). Every kernel of the old build must exist in the new one with the same
instruction text and the same registers, stack, static shared memory and local memory (a template kernel instantiated in several translation units has one
copy per unit: the copies are compared as a set); kernels only the new build has are listed. Exit status 0 when nothing
changed, 1 otherwise.
"""
from __future__ import annotations

import argparse
import os
import re
import shutil
import subprocess
import sys
from typing import Dict, List, Tuple

_FUNC = re.compile(r"^\s*Function : (\S+)\s*$")
_RES = re.compile(r"^\s*Function (\S+):\s*$")
_KEEP = re.compile(r"\b(REG|STACK|SHARED|LOCAL):(\d+)")   # the parameter bank (CONSTANT[0]) grows with a new parameter


def _cuobjdump() -> str:
    exe = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    if not os.path.exists(exe):
        sys.exit("cuobjdump not found (put the CUDA toolkit's bin directory on PATH or set CUDA_HOME)")
    return exe


def _run(args: List[str]) -> str:
    return subprocess.run(args, check=True, capture_output=True, text=True).stdout


def demangle(names: List[str]) -> Dict[str, str]:
    if not names:
        return {}
    exe = shutil.which("cu++filt") or shutil.which("c++filt")
    if exe is None:
        sys.exit("c++filt not found")
    out = subprocess.run([exe], input="\n".join(names) + "\n", check=True, capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))


def kernel_key(demangled: str) -> str:
    """Qualified name + template arguments: the return type and the trailing parameter list are dropped."""
    s = demangled.strip()
    if s.endswith(")"):                                  # strip the balanced (...) at the end: the parameter list
        depth = 0
        for i in range(len(s) - 1, -1, -1):
            depth += s[i] == ")"
            depth -= s[i] == "("
            if depth == 0:
                s = s[:i]
                break
    if s.startswith("void "):
        s = s[5:]
    return s.strip()


def drop_trailing_false(key: str) -> str:
    """``k<a, b, false>`` -> ``k<a, b>``, ``k<false>`` -> ``k``; anything else unchanged (cu++filt spells false
    ``(bool)0``, c++filt ``false``)."""
    for f in ("false", "(bool)0"):
        if key.endswith(f", {f}>"):
            return key[: -len(f", {f}>")] + ">"
        if key.endswith(f"<{f}>"):
            return key[: -len(f"<{f}>")]
    return key


def _normalise(line: str) -> str:
    return re.sub(r"\s+", " ", line).strip()


Kernel = Tuple[Tuple[str, ...], str]                    # (instruction lines, "REG:n STACK:n SHARED:n LOCAL:n") of one copy


def read_library(path: str) -> Dict[str, List[Kernel]]:
    """kernel key -> its copies, sorted"""
    exe = _cuobjdump()
    sass = _run([exe, "-sass", path]).splitlines()
    res = _run([exe, "-res-usage", path]).splitlines()
    bodies: List[Tuple[str, List[str]]] = []              # in file order; cuobjdump lists -sass and -res-usage alike
    for line in sass:
        m = _FUNC.match(line)
        if m:
            bodies.append((m.group(1), []))
            continue
        if bodies and line.strip().startswith("/*") and "*/" in line:
            bodies[-1][1].append(_normalise(line))
    regs: Dict[str, List[str]] = {}
    for line, nxt in zip(res, res[1:] + [""]):          # "Function <name>:" then its resource line
        m = _RES.match(line)
        if m:
            regs.setdefault(m.group(1), []).append(" ".join(f"{a}:{b}" for a, b in _KEEP.findall(nxt)))
    names = demangle(sorted({n for n, _ in bodies}))
    out: Dict[str, List[Kernel]] = {}
    seen: Dict[str, int] = {}
    for mangled, body in bodies:
        i = seen.get(mangled, 0)
        seen[mangled] = i + 1
        reg = regs.get(mangled, [])
        if i >= len(reg):
            sys.exit(f"{path}: no resource usage listed for {mangled}")
        out.setdefault(kernel_key(names[mangled]), []).append((tuple(body), reg[i]))
    return {k: sorted(v) for k, v in out.items()}


def compare(old: Dict[str, List[Kernel]], new: Dict[str, List[Kernel]]) -> Tuple[List[str], List[str], List[str]]:
    """(report lines, problems, kernels only in the new build)"""
    alias: Dict[str, str] = {}
    for k in new:
        d = drop_trailing_false(k)
        if d != k and d not in new:
            alias[d] = k
    report, problems, used = [], [], set()
    for k in sorted(old):
        nk = k if k in new else alias.get(k)
        if nk is None:
            problems.append(f"MISSING   {k}")
            continue
        used.add(nk)
        oc, nc = old[k], new[nk]
        if [b for b, _ in oc] != [b for b, _ in nc]:
            ob, nb = oc[0][0], nc[0][0]
            diff = next((i for i, (a, b) in enumerate(zip(ob, nb)) if a != b), min(len(ob), len(nb)))
            problems.append(f"CHANGED   {k}: {len(oc)} -> {len(nc)} copies, {len(ob)} -> {len(nb)} instructions, "
                            f"first difference at instruction {diff}")
        elif [r for _, r in oc] != [r for _, r in nc]:
            problems.append(f"RESOURCES {k}: {[r for _, r in oc]} -> {[r for _, r in nc]}")
        else:
            report.append(f"same      {k}" + (f"  (as {nk})" if nk != k else "") +
                          f"  [{len(oc[0][0])} instructions, {oc[0][1]}, {len(oc)} cop{'y' if len(oc) == 1 else 'ies'}]")
    added = sorted(k for k in new if k not in used)
    return report, problems, added


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("old", help="libmarlsc_b200.so of the older build")
    ap.add_argument("new", help="libmarlsc_b200.so of the newer build")
    ap.add_argument("--verbose", action="store_true", help="list every unchanged kernel")
    a = ap.parse_args()
    old, new = read_library(a.old), read_library(a.new)
    report, problems, added = compare(old, new)
    if a.verbose:
        print("\n".join(report))
    for k in added:
        print(f"new       {k}  [{len(new[k][0][0])} instructions, {new[k][0][1]}]")
    for p in problems:
        print(p)
    print(f"{len(old)} kernels in the old build: {len(report)} unchanged, {len(problems)} changed or missing; "
          f"{len(added)} new kernels")
    return 1 if problems else 0


if __name__ == "__main__":
    sys.exit(main())
