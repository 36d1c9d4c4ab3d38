"""Code layout of the NUTS kernels (development tool): where each region of mdg_nuts_kernel.cuh sits in the SASS.

    python tools/sass_layout.py [LIB.so | X.cubin] [--source mdg_nuts_kernel.cuh] [--min-run 24]

The library (default: the in-tree build) or a cubin built from nuts_group_kernel<MODEL, 8, 4> is disassembled with
`nvdisasm -gi` (line information with the inlining chain; the build's `-lineinfo` provides it). Each instruction of
a kernel is given to the outermost frame of its chain that lies in the kernel source (`--source`, matched by file
name: the line in the kernel that the code was inlined into), and that line to a region by the REGION MARKERS of the source: a comment `layout: NAME` starts region NAME at
its line, and the region runs to the next marker. Code inlined from other headers or from helpers
and lambdas of the kernel source (the evaluation, the special functions) thus counts for the kernel line that calls it. Functions the kernel calls out of line (`__noinline__`, `MDG_COLD`, the
CUDA math library's slow paths) are emitted after the kernel's body in the same section; they are listed by name.
ptxas also emits, at the end of the body, a divergent copy of every group-masked shuffle (`WARPSYNC.COLLECTIVE` ...
`ENDCOLLECTIVE`), run only when a group reaches the shuffle with some of its own lanes inactive; from the basic block
of the first `WARPSYNC.COLLECTIVE` on, the body is counted as the cold region `divergent_shuffles`.

Every region is warm (run on every leapfrog or every transition) or cold (once per chain, once per adaptation window,
rare fallbacks, optional stores); WARM below lists the warm ones. For each kernel the tool prints
  * the body in address order as runs of one region (runs shorter than --min-run instructions are folded into the
    run before them and counted in its `mixed` column),
  * the warm span: from the first to the last instruction of a warm region, and the cold instructions inside it,
  * the instructions per region and the out-of-line functions.
One instruction is 16 bytes."""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_SOURCE = os.path.join(ROOT, "metadamage_b200", "csrc", "mdg_nuts_kernel.cuh")
WARM = ("eval", "head", "leaf", "subtree_end", "transition_end", "adapt", "kept_draw", "transition_start", "doubling")
CUDA = "/usr/local/cuda/bin"

FRAME = re.compile(r'File "([^"]+)", line (\d+)')
INSN = re.compile(r"^\s+/\*([0-9a-f]+)\*/\s+(\S.*?)\s*;?\s*$")
LABEL = re.compile(r"^(\S+):\s*$")


def tool(name):
    path = os.path.join(CUDA, name)
    return path if os.path.exists(path) else name


def cubins(path, tmp):
    if path.endswith(".cubin"):
        return [path]
    subprocess.run([tool("cuobjdump"), "-xelf", "all", os.path.abspath(path)], cwd=tmp, check=True, capture_output=True)
    return [os.path.join(tmp, f) for f in sorted(os.listdir(tmp)) if f.endswith(".cubin")]


def markers(source):
    """[(first line, region)] in line order, from the `layout: NAME` comments of the kernel source."""
    out = []
    with open(source) as f:
        for i, line in enumerate(f, 1):
            m = re.search(r"//.*\blayout: ([a-z_]+)", line)
            if m:
                out.append((i, m.group(1)))
    if not out:
        sys.exit(f"{source}: no `layout: NAME` markers")
    return out


def region_of(line, marks):
    name = "(before the first marker)"
    for first, reg in marks:
        if first > line:
            break
        name = reg
    return name


def kernels(disasm, src_name, marks):
    """{kernel: (body [(address, region)], {out-of-line function: instructions})}"""
    out, kern, sub, frames, fresh, block, tail = {}, None, None, [], True, 0, None
    for line in disasm.splitlines():
        m = re.match(r"\s*\.section\s+\.text\.(\S+?),", line)
        if m:
            kern = m.group(1) if "nuts_group_kernel" in m.group(1) else None
            sub, frames, tail = None, [], None
            if kern:
                out[kern] = ([], collections.Counter())
            continue
        if kern is None:
            continue
        m = LABEL.match(line)
        if m and m.group(1).startswith("$"):
            sub = m.group(1).split("$")[-1] or m.group(1)
            continue
        if m:
            block = len(out[kern][0])
        if line.lstrip().startswith("//##"):
            chain = FRAME.findall(line)
            # several //## lines may precede one instruction (the one with the longest chain is the most precise);
            # an instruction without one continues the line before it
            if fresh or len(chain) >= len(frames):
                frames = chain
            fresh = False
            continue
        m = INSN.match(line)
        if not m:
            continue
        body, subs = out[kern]
        if sub is not None:
            subs[sub] += 1
        else:
            own = [int(ln) for fn, ln in frames if os.path.basename(fn) == src_name]
            body.append((int(m.group(1), 16), region_of(own[-1], marks) if own else "(no line in the source)"))
            if "WARPSYNC.COLLECTIVE" in m.group(2) and tail is None:
                tail = block
            if tail is not None:
                body[tail:] = [(a, "divergent_shuffles") for a, _ in body[tail:]]
        fresh = True
    return out


def demangle(name):
    r = subprocess.run(["c++filt", name], capture_output=True, text=True)
    return (r.stdout.strip() or name).split("(")[0]


def report(name, body, subs, min_run):
    print(f"## `{demangle(name)}`\n")
    n = len(body)
    print(f"{n} instructions in the kernel body, {sum(subs.values())} in {len(subs)} out-of-line functions "
          f"({n * 16 / 1024:.1f} KB + {sum(subs.values()) * 16 / 1024:.1f} KB)\n")
    runs = []  # [region, first index, last index, mixed]
    for i, (_, reg) in enumerate(body):
        if runs and runs[-1][0] == reg:
            runs[-1][2] = i
        else:
            runs.append([reg, i, i, 0])
    folded = []
    for r in runs:
        length = r[2] - r[1] + 1
        if folded and (length < min_run or folded[-1][0] == r[0]):
            folded[-1][2] = r[2]
            folded[-1][3] += 0 if folded[-1][0] == r[0] else length
        else:
            folded.append(list(r))
    print("| instructions | region | warm | mixed |")
    print("|---|---|---|---|")
    for reg, a, b, mixed in folded:
        print(f"| {a}–{b + 1} | {reg} | {'yes' if reg in WARM else ''} | {mixed or ''} |")
    warm_idx = [i for i, (_, reg) in enumerate(body) if reg in WARM]
    if warm_idx:
        a, b = warm_idx[0], warm_idx[-1]
        inside = collections.Counter(reg for _, reg in body[a:b + 1] if reg not in WARM)
        print(f"\nwarm span: instructions {a}–{b + 1} = {b + 1 - a} instructions ({(b + 1 - a) * 16 / 1024:.1f} KB), "
              f"of which {len(warm_idx)} warm and {sum(inside.values())} not")
        if inside:
            print("cold inside the warm span: " + ", ".join(f"{reg} {c}" for reg, c in inside.most_common()))
    per = collections.Counter(reg for _, reg in body)
    print("\n| region | instructions | warm |\n|---|---|---|")
    for reg, c in per.most_common():
        print(f"| {reg} | {c} | {'yes' if reg in WARM else ''} |")
    if subs:
        print("\n| out-of-line function | instructions |\n|---|---|")
        for s, c in subs.most_common():
            print(f"| `{demangle(s)}` | {c} |")
    print()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("binary", nargs="?", default=os.path.join(ROOT, "metadamage_b200", "libmdgb200.so"))
    ap.add_argument("--source", default=DEFAULT_SOURCE, help="the kernel source the binary was built from, with region markers")
    ap.add_argument("--min-run", type=int, default=24)
    args = ap.parse_args()
    marks = markers(args.source)
    with tempfile.TemporaryDirectory() as tmp:
        found = {}
        for cub in cubins(args.binary, tmp):
            dis = subprocess.run([tool("nvdisasm"), "-gi", cub], capture_output=True, text=True, check=True).stdout
            for k, v in kernels(dis, os.path.basename(args.source), marks).items():
                found.setdefault(k, v)
    if not found:
        sys.exit(f"{args.binary}: no nuts_group_kernel")
    print(f"# SASS layout of the NUTS kernels: `{os.path.basename(args.binary)}`, regions of `{os.path.basename(args.source)}`\n")
    for k in sorted(found):
        report(k, *found[k], args.min_run)


if __name__ == "__main__":
    main()
