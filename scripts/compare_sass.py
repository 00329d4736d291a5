"""Compare the device code of two builds of libbrl_b200.so kernel by kernel.

    python scripts/compare_sass.py OLD.so NEW.so [--out report.txt]

For every kernel of OLD it finds the kernel of NEW that plays the same role and compares the SASS (instruction text and
encodings, `cuobjdump -sass`) and the resources (`cuobjdump -res-usage`: registers, stack, shared and local memory, and the
constant bank that holds the parameter block).  A refactor that changes template parameter lists changes the mangled names,
so kernels are paired by their demangled names after the renames in RENAMES; a rename to None marks a kernel the change
removes on purpose.  Exit status 0 when every remaining kernel is identical and nothing else appeared or disappeared.

RENAMES and ADDED record the SMC hand-reading change (DESIGN.md f19): f18's segment-count and public-pass kernels became
templates over the row set a forward reads, and f18's own row set (every call of the prefix) is the empty instantiation;
the SMC kernels (brl::k_smc_*) and the SmcWindow instantiations are added.  Replace both tables for another change."""
import argparse
import os
import re
import subprocess
import sys
from collections import OrderedDict

# (pattern, replacement) on names demangled as cu++filt prints them: template arguments read (int)128, (bool)1
RENAMES = [(r"^brl::k_post_count$", "brl::k_post_count<>"),
           (r"^brl::k_post_public$", "brl::k_post_public<>")]
ADDED = [r"^brl::k_smc_", r"^brl::k_post_(count|public)<brl::SmcWindow>$"]  # patterns of kernels the change adds on purpose: reported, not counted as unexpected


def _cuobjdump(flag, lib):
    return subprocess.run(["cuobjdump", flag, lib], check=True, capture_output=True, text=True).stdout


def _demangle(names):
    out = subprocess.run(["cu++filt"], input="\n".join(names), check=True, capture_output=True, text=True).stdout.splitlines()
    short = []
    for d in out:
        depth = 0
        for i, ch in enumerate(d):  # the parameter list opens at the first '(' outside the template arguments
            depth += (ch == "<") - (ch == ">")
            if ch == "(" and depth == 0:
                d = d[:i]
                break
        short.append(d[5:] if d.startswith("void ") else d)
    return dict(zip(names, short))


def _split(text, head):
    """{(translation unit, mangled name): body} of every function in a cuobjdump listing; `head` matches a function's line"""
    funcs, tu, cur = OrderedDict(), "?", None
    for line in text.splitlines():
        m = re.match(r"\s*identifier = (.*)", line)
        if m:
            tu, cur = os.path.basename(m.group(1).strip()), None
            continue
        m = re.match(head, line)
        if m:
            cur = (tu, m.group(1))
            funcs[cur] = []
            continue
        if line.startswith("Fatbin"):
            cur = None
        elif cur is not None and line.strip():
            funcs[cur].append(" ".join(line.split()))  # cuobjdump pads columns to the listing's longest line
    return funcs


def kernels(lib):
    """{(translation unit, demangled name): (sass lines, resource line)}"""
    sass = _split(_cuobjdump("-sass", lib), r"\s*Function : (\S+)")
    res = _split(_cuobjdump("-res-usage", lib), r"\s*Function (\S+):$")
    names = _demangle(sorted({n for _, n in sass}))
    out = {}
    for (tu, n), body in sass.items():
        key = (tu, names[n])
        if key in out:
            raise SystemExit(f"{lib}: two kernels named {key}")
        out[key] = (body, " ".join(res.get((tu, n), ["?"])))
    return out


def renamed(name):
    for pat, rep in RENAMES:
        if re.match(pat, name):
            return None if rep is None else re.sub(pat, rep, name)
    return name


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--out", help="also write the report here")
    a = ap.parse_args(argv)
    old, new = kernels(a.old), kernels(a.new)
    lines, bad, removed, same = [], 0, 0, 0
    matched = set()
    for (tu, name), (body, res) in sorted(old.items()):
        target = renamed(name)
        if target is None:
            removed += 1
            lines.append(f"removed    {tu}  {name}  [{res}]")
            continue
        got = new.get((tu, target))
        if got is None:
            bad += 1
            lines.append(f"MISSING    {tu}  {name} -> {target}")
            continue
        matched.add((tu, target))
        if got[0] == body and got[1] == res:
            same += 1
            lines.append(f"identical  {tu}  {name} -> {target}  ({sum(1 for x in body if re.match(r'/\*[0-9a-f]+\*/', x))} instructions)  [{res}]")
        else:
            bad += 1
            what = "SASS" if got[0] != body else "resources"
            lines.append(f"DIFFERENT  {tu}  {name} -> {target}  ({what})  old [{res}] new [{got[1]}]")
    added = 0
    for key in sorted(set(new) - matched):
        if any(re.match(pat, key[1]) for pat in ADDED):
            added += 1
            lines.append(f"added      {key[0]}  {key[1]}  [{new[key][1]}]")
        else:
            bad += 1
            lines.append(f"ADDED      {key[0]}  {key[1]}  [{new[key][1]}]")
    lines.append(f"{len(old)} kernels before, {len(new)} after: {same} identical, {removed} removed as intended, {added} added as intended, "
                 f"{bad} unexpected")
    report = "\n".join(lines) + "\n"
    sys.stdout.write(report)
    if a.out:
        with open(a.out, "w") as f:
            f.write(report)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
