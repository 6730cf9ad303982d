"""Static instruction census of the integration kernel's fast path (CPU only, no GPU needed).

Disassembles integrate_kernel<2> (the default z-split) with source-line information and prints the
opcode tally of one 8-voxel group on the fast path: the branch-free projection, the gathers and the
record updates of one frame of one column, with the column set-up before them left out.  The group
is taken from the SASS, not from the source: every instruction from the first one of the fast
projection block (`if (fast) {` in volume.cu) to the conditional backward branch that closes the
frame loop, minus
  - the address range of the IEEE projection block (the `else` of `if (fast)`), and
  - every instruction whose line chain (inlined call sites included) passes through a source line
    that calls __fdiv_rn: the IEEE division fallback, per lane or per warp.
Reconvergence barriers (BSSY/BSYNC), CALLs and constant-bank reloads (LDCU) left in that body are the
control-flow and parameter overhead the update path pays per group.

    python tools/k4_sass_census.py                    # the built library (libotslam_b200.so)
    python tools/k4_sass_census.py --compile          # nvcc -c csrc/volume.cu into a temporary directory
    python tools/k4_sass_census.py --obj volume.o     # any object / cubin / library holding the kernel
"""
import argparse
import collections
import glob
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "object-triggered-3d-slam_b200")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
KERNEL = "_ZN6otslam16integrate_kernelILi2EEEvNS_13IntegrateArgsE"
LINE_RE = re.compile(r'//## File "([^"]+)", line (\d+)((?: inlined at "[^"]+", line \d+)*)')
INL_RE = re.compile(r'inlined at "([^"]+)", line (\d+)')
INS_RE = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def compile_volume(tmp):
    sys.path.insert(0, PKG)
    import build  # the library's own flags
    obj = os.path.join(tmp, "volume.o")
    subprocess.check_call([build.NVCC] + build.FLAGS + ["-c", os.path.join(PKG, "csrc", "volume.cu"), "-o", obj])
    return obj


def disassemble(path, tmp):
    """nvdisasm -gi of the cubin holding KERNEL, restricted to that kernel's text section."""
    if path.endswith(".cubin"):
        cubins = [path]
    else:
        subprocess.check_call([os.path.join(CUDA, "bin", "cuobjdump"), "-xelf", "all", os.path.abspath(path)], cwd=tmp,
                              stdout=subprocess.DEVNULL)
        cubins = sorted(glob.glob(os.path.join(tmp, "*.cubin")))
    for c in cubins:
        out = subprocess.run([os.path.join(CUDA, "bin", "nvdisasm"), "-gi", c], check=True, capture_output=True,
                             text=True).stdout
        start = out.find(".text." + KERNEL + ":")
        if start >= 0:
            end = out.find("//---------------------", start)
            return out[start:end if end > 0 else len(out)]
    raise SystemExit(f"{KERNEL} not found in {path}")


def parse(text):
    """[(address, instruction text, line chain [(file, line), ...] innermost first)], {label: address}"""
    chain, ins, labels, pending, fresh = [], [], {}, [], True
    for raw in text.splitlines():
        m = LINE_RE.search(raw)
        if m:   # consecutive annotations describe one position: the inlined line, then each call site
            chain = ([] if fresh else chain) + [(m.group(1), int(m.group(2)))] + \
                [(f, int(n)) for f, n in INL_RE.findall(m.group(3))]
            fresh = False
            continue
        m = re.match(r"^(\.L_x_\d+):", raw)
        if m:
            pending.append(m.group(1))
            continue
        m = INS_RE.search(raw)
        if m:
            a = int(m.group(1), 16)
            labels.update((p, a) for p in pending)
            pending, fresh = [], True
            ins.append((a, m.group(2), chain))
    return ins, labels


def branch_target(text, labels):
    m = re.search(r"`\((\.L_x_\d+)\)", text)
    return labels.get(m.group(1)) if m else None


def block_end(lines, i):
    """index of the line closing the block that line i opens (line i may be `} else {`)"""
    depth = 1
    for k in range(i + 1, len(lines)):
        depth += lines[k].count("{") - lines[k].count("}")
        if depth <= 0:
            return k
    raise ValueError("unbalanced braces")


def source_marks(src):
    """1-based line numbers: fast block [start, else), IEEE block [else, else_end], __fdiv_rn lines"""
    lines = open(src).read().splitlines()
    k4 = next(i for i, l in enumerate(lines) if "integrate_kernel(IntegrateArgs" in l)
    fast = next(i for i in range(k4, len(lines)) if re.match(r"\s*if \(fast\) \{", lines[i]))
    els = next(i for i in range(fast, len(lines)) if re.match(r"\s*\} else \{", lines[i]))
    els_end = block_end(lines, els)
    fdiv = {i + 1 for i, l in enumerate(lines) if "__fdiv_rn(" in l and not l.lstrip().startswith("//")}
    return fast + 1, els + 1, els_end + 1, fdiv


def opcode(text):
    t = re.sub(r"^@!?U?P\w+\s+", "", text)
    return t.split()[0]


def census(path):
    with tempfile.TemporaryDirectory() as tmp:
        if path is None:
            path = compile_volume(tmp)
        ins, labels = parse(disassemble(path, tmp))
    src = next(f for _, _, ch in ins for f, _ in ch if f.endswith("volume.cu"))
    fast, els, els_end, fdiv = source_marks(src)

    def at(ch, lo, hi):
        return any(f == src and lo <= n <= hi for f, n in ch)

    # the frame loop closes with the conditional backward branch of widest span
    back = max((k for k, (a, t, _) in enumerate(ins) if t.startswith("@") and opcode(t) == "BRA"
                and (branch_target(t, labels) or a) < a), key=lambda k: ins[k][0] - branch_target(ins[k][1], labels))
    head = branch_target(ins[back][1], labels)
    # fast projection entry: the first fast-block instruction inside the loop that follows a branch (the column guard's)
    first = next(k for k in range(1, back) if ins[k][0] > head and at(ins[k][2], fast + 1, els - 1)
                 and opcode(ins[k - 1][1]) == "BRA")
    slow = [a for a, _, ch in ins[first:back] if at(ch, els + 1, els_end - 1)]
    slo, shi = (min(slow), max(slow)) if slow else (-1, -1)
    body = [(a, t) for a, t, ch in ins[first:back + 1]
            if not (slo <= a <= shi) and not any(f == src and n in fdiv for f, n in ch)]
    return path, body


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--obj", help="object, cubin or shared library holding integrate_kernel<2>")
    ap.add_argument("--compile", action="store_true", help="compile csrc/volume.cu with the library's flags")
    ap.add_argument("--list", action="store_true", help="also print the body's instructions")
    args = ap.parse_args()
    path = None if args.compile else (args.obj or os.path.join(PKG, "libotslam_b200.so"))
    label = path or "csrc/volume.cu (compiled)"
    _, body = census(path)
    tally = collections.Counter(opcode(t) for _, t in body)
    print(f"integrate_kernel<2>, fast-path 8-voxel group body, from {label}")
    if args.list:
        for a, t in body:
            print(f"  {a:05x}  {t}")
    print(f"instructions: {len(body)}  ({len(body) / 8:.1f} per voxel)")
    for key in ("BSSY", "BSYNC", "CALL", "LDCU", "BRA", "VOTE", "SEL"):
        n = sum(v for k, v in tally.items() if k.split(".")[0] == key)
        print(f"  {key:6s} {n}")
    print("opcode tally:")
    for k, v in sorted(tally.items(), key=lambda kv: (-kv[1], kv[0])):
        print(f"  {k:28s} {v}")


if __name__ == "__main__":
    main()
